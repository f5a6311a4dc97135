// Kernels and C-ABI of the batched four-player-chess environment (sm_100a).
// See include/fpc.h for the boundary and fpc_device.cuh for the rules.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/fpc.h"
#include "fpc_host.h"
#include "fpc_rules.cuh"

namespace fpc {

constexpr int WARPS_PER_BLOCK = 4;  // one warp per game
constexpr int BLOCK_THREADS = WARPS_PER_BLOCK * 32;

// Dense outputs.  The reference tensors are dense f32 ([n,24,R,R] planes, [n,8R+8,R,R] mask) holding
// ~40 and ~19-38 ones per game among 4,704 and 23,520 cells; writing them is the HBM-bound part of the
// path (113 KB per game at 14x14).  rules_kernel produces them as two short records per game -- the plane cells
// and the flat action indices that are 1.0 (fpc_rules.cuh: CELL_* / FLAT_*) -- and expand_kernel streams the
// tensors out: zero fill, then the ones.  The two kernels run on different streams so that the expansion of one
// batch overlaps the integer work of the next (FPC_FLAG_ASYNC_DENSE, fpc_join).

static_assert(STATUS_IN_CHECK == FPC_STATUS_IN_CHECK && STATUS_CAN_TAKE_KING == FPC_STATUS_CAN_TAKE_KING &&
                  STATUS_OVERFLOW == FPC_STATUS_OVERFLOW && STATUS_FINISHED == FPC_STATUS_FINISHED &&
                  STATUS_CHECK == FPC_STATUS_CHECK,
              "status bits of fpc_rules.cuh and include/fpc.h");

// The rules kernel: one warp per game (fpc_rules.cuh).  Legal moves, result, the bit sets of the dense outputs,
// and (playout) the move choice and make-move.  It touches only the board store and compact per-game outputs.
template <class G>
__global__ void __launch_bounds__(BLOCK_THREADS) rules_kernel(const __grid_constant__ ObserveParams P) {
  __shared__ RulesScratch<G> scratch[WARPS_PER_BLOCK];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * WARPS_PER_BLOCK + wib;
  if (g >= P.n) return;
  rules_warp<G>(P, scratch[wib], g, lane);
}

// Records -> dense f32 (0.0 / 1.0).  A persistent kernel, ONE CTA per SM, each CTA taking every gridDim.x-th game:
// the records of the game are requested first, then every thread streams zeros over the game's two tensors (coalesced
// 16-byte st.global.cs, nothing to wait for: the stores do not depend on any load), the CTA synchronises, and one
// thread per recorded one writes its 1.0f.  The ones land in lines this CTA has just written, so they merge in L2 and
// HBM sees each line once.  ~10 instructions per 512-byte store instruction and only 12 warps per SM: measured on
// B200 (tools/overlap_probe.py, DESIGN.md) a grid that floods the SMs with store warps streams a little faster alone
// (69-71 us vs 73 us per 462 MB) but loses twice that when the rules kernel of the next step shares the SMs, because
// every shared-memory / global access of the rules warps queues behind the stores in the load/store pipe.
// HBM-write bound.
constexpr int EXPAND_THREADS = 384;

template <class G>
__global__ void __launch_bounds__(EXPAND_THREADS)
    expand_kernel(const uint16_t *__restrict__ cells, float *__restrict__ planes, const uint16_t *__restrict__ flats,
                  float *__restrict__ mask, int n) {
  constexpr int P4 = G::SSZ / 4, M4 = G::ASZ / 4;
  const int t = threadIdx.x, T = blockDim.x;
  const float4 zero = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  for (int game = blockIdx.x; game < n; game += gridDim.x) {
    const uint16_t *gc = planes ? cells + (size_t)game * CELL_STRIDE : nullptr;
    const uint16_t *gf = mask ? flats + (size_t)game * FLAT_STRIDE : nullptr;
    // the records are requested first and travel while the zeros are written
    const int n_cells = gc ? gc[0] : 0, n_flats = gf ? gf[0] : 0;
    const int my_cell = t < n_cells ? gc[CELL_FIRST + t] : -1;
    const int my_flat = t < n_flats ? gf[FLAT_FIRST + t] : -1;
    float *pl = planes + (size_t)game * G::SSZ, *mk = mask + (size_t)game * G::ASZ;
    if (planes)
      for (int i = t; i < P4; i += T) __stcs(reinterpret_cast<float4 *>(pl) + i, zero);
    if (mask)
      for (int i = t; i < M4; i += T) __stcs(reinterpret_cast<float4 *>(mk) + i, zero);
    __syncthreads();  // block-wide memory ordering: every zero precedes every one
    if (my_cell >= 0) pl[my_cell] = 1.0f;
    if (my_flat >= 0) mk[my_flat] = 1.0f;
    for (int i = t + T; i < n_cells; i += T) pl[gc[CELL_FIRST + i]] = 1.0f;
    for (int i = t + T; i < n_flats; i += T) mk[gf[FLAT_FIRST + i]] = 1.0f;
  }
}

// chess::Board::MakeMove (engine/board.cpp:1028-1096) for arbitrary 8-byte moves, or for
// index-built moves (src/cpp/move.cpp:41-61) when flat != null.  Works on the record bytes.
template <class G>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
    make_kernel(const uint8_t *in, const uint64_t *moves, const int32_t *flat, int n, uint8_t *out, int32_t *err) {
  __shared__ alignas(16) uint8_t recs[WARPS_PER_BLOCK][256];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * WARPS_PER_BLOCK + wib;
  if (g >= n) return;
  uint8_t *b = recs[wib];
  if (lane < G::REC / 16)
    reinterpret_cast<uint4 *>(b)[lane] = reinterpret_cast<const uint4 *>(in + (size_t)g * G::REC)[lane];
  __syncwarp();
  if (lane == 0) {
    constexpr int NSQ = G::NSQ;
    int from, to, promo = NO_PIECE, rf = NSQ, rt = NSQ;
    uint32_t r1 = 0;
    if (flat) {
      decode_flat_move<G>(flat[g], from, to);
    } else {
      const uint64_t m = moves[g];
      from = (int)(m & 0xff);
      to = (int)((m >> 8) & 0xff);
      promo = (int)((m >> 24) & 0xff);
      rf = (int)((m >> 32) & 0xff);
      rt = (int)((m >> 40) & 0xff);
      r1 = (uint32_t)((m >> 56) & 0xff);
    }
    const int code = apply_move_record<G>(b, from, to, promo, rf, rt, r1) ? FPC_OK : FPC_ERR_MOVE;
    if (err) err[g] = code;
  }
  __syncwarp();
  if (lane < G::REC / 16)
    reinterpret_cast<uint4 *>(out + (size_t)g * G::REC)[lane] = reinterpret_cast<const uint4 *>(b)[lane];
}

// chess::Board::CalculateHeuristic (engine/board.cpp:1263-1292) for the team to move.
template <class G>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32) heuristic_kernel(const uint8_t *in, int n, int32_t *value) {
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * WARPS_PER_BLOCK + wib;
  if (g >= n) return;
  const uint8_t *b = in + (size_t)g * G::REC;
  const int team = b[G::OFF_TURN] & 1;
  int h = 0;
  for (int sq = lane; sq < G::NSQ; sq += 32) {
    const uint32_t p = b[sq];
    if (present(p) && type_of(p) != KING) {
      const int t = type_of(p);
      const int v = t == PAWN ? 1 : (t == ROOK ? 5 : (t == QUEEN ? 9 : 3));
      h += team_of(p) == team ? v : -v;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) h += __shfl_xor_sync(FULL, h, o);
  if (lane == 0) value[g] = h;
}

// ---- host side ----------------------------------------------------------------------------

static thread_local std::string g_err;

int fail(int code, const std::string &msg) {
  g_err = msg;
  return code;
}
int cuda_check(cudaError_t e, const char *what) {
  if (e == cudaSuccess) return FPC_OK;
  return fail(FPC_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

// One record pair (plane cells / mask flats) per game, double-buffered: rules_kernel of a full rewrite writes one half
// while expand_kernel of an earlier call may still read the other.  cur_*: the half with the tensor's latest record.
struct Records {
  uint16_t *cells[2] = {nullptr, nullptr}, *flats[2] = {nullptr, nullptr};
  size_t games = 0;
  int cur_cells = 0, cur_flats = 0;
  int release() {
    for (int i = 0; i < 2; ++i) {
      cudaFree(cells[i]);
      cudaFree(flats[i]);
      cells[i] = flats[i] = nullptr;
    }
    games = 0;
    return FPC_OK;
  }
  int reserve(size_t n) {
    if (n <= games) return FPC_OK;
    release();
    for (int i = 0; i < 2; ++i) {
      CK(cudaMalloc(&cells[i], n * CELL_STRIDE * sizeof(uint16_t)));
      CK(cudaMalloc(&flats[i], n * FLAT_STRIDE * sizeof(uint16_t)));
    }
    games = n;
    return FPC_OK;
  }
};

// Optional CUDA-event timing of one dense call's two launches on their own streams (fpc_profile_enable / _read).
struct LaunchTimes {
  cudaEvent_t rules[2], expand[2];  // start, stop
};
constexpr int PROF_MAX = 4096;

// Per host thread and device: the streams the two kernels of a dense call run on, their events, and the records of
// calls without a fpc_dense_track.
struct DeviceState {
  int device = -1;
  int sms = 0;                  // multiprocessors: the grid of expand_kernel
  cudaStream_t side = nullptr;  // expand_kernel: lowest priority
  cudaStream_t hi = nullptr;    // rules_kernel when dense outputs are wanted: highest priority, so that its
                                // CTAs are dispatched ahead of the remaining CTAs of a running expansion
  cudaEvent_t fork = nullptr;
  cudaEvent_t rules_done[2] = {nullptr, nullptr}, expand_done[2] = {nullptr, nullptr};
  // expand_done[b] is whichever of these two was recorded last for slot b: the plain one (no timing) in steady state,
  // the timestamped one while a pipeline of dense calls is starting up (end_event)
  cudaEvent_t expand_done_plain[2] = {nullptr, nullptr}, expand_done_stamped[2] = {nullptr, nullptr};
  int startup_left = 0;
  bool expand_recorded[2] = {false, false};
  int parity = 0;           // event slot of the next full rewrite
  int last = -1;            // event slot of the most recent expansion (fpc_join)
  bool last_async = false;  // ... which the caller's stream has not been made to wait for (FPC_FLAG_ASYNC_DENSE)
  unsigned carveout_set = 0;  // bit R: the shared-memory carveout of board size R's two kernels is requested
  Records ws;
  bool prof_on = false;
  int prof_n = 0;
  std::vector<LaunchTimes> prof;
};
constexpr int MAX_DEVICES = 16;
static thread_local DeviceState g_dev[MAX_DEVICES];

// The calling thread's state on the current device.  With `create`, its streams and events are made on first use.
static int device_state(DeviceState **out, bool create) {
  int dev = 0;
  CK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= MAX_DEVICES) return fail(FPC_ERR_ARG, "device ordinal out of range");
  DeviceState &S = g_dev[dev];
  if (create && !S.side) {
    S.device = dev;
    CK(cudaDeviceGetAttribute(&S.sms, cudaDevAttrMultiProcessorCount, dev));
    int least = 0, greatest = 0;
    CK(cudaDeviceGetStreamPriorityRange(&least, &greatest));
    CK(cudaStreamCreateWithPriority(&S.side, cudaStreamNonBlocking, least));
    CK(cudaStreamCreateWithPriority(&S.hi, cudaStreamNonBlocking, greatest));
    CK(cudaEventCreateWithFlags(&S.fork, cudaEventDisableTiming));
    for (int i = 0; i < 2; ++i) {
      CK(cudaEventCreateWithFlags(&S.rules_done[i], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&S.expand_done_plain[i], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&S.expand_done_stamped[i], cudaEventDefault));
      S.expand_done[i] = S.expand_done_plain[i];
    }
  }
  *out = &S;
  return FPC_OK;
}

}  // namespace fpc

// Explicit handle for resident dense tensors (FPC_FLAG_INCREMENTAL): it owns the records of the ones the latest dense
// call through it left in ONE planes tensor and / or ONE mask tensor.  Nothing is keyed on pointer identity alone: a
// handle only vouches for tensors it was itself used with since its creation or last invalidation.
struct fpc_dense_track {
  unsigned magic;
  int device, R, n;
  fpc::Records rec;
  // per tensor: the pointer the record describes, whether the content is known
  const float *planes, *mask;
  bool known_planes, known_mask;
};

namespace fpc {
constexpr unsigned TRACK_MAGIC = 0x46504354u;  // "FPCT"

struct DenseOut {
  float *planes, *mask;
  int flags;
  fpc_dense_track *track;
};

// Incremental update: the tensors hold exactly the recorded ones, so the rules kernel clears those and sets the new
// ones on the caller's stream, with no expansion.  A still running expansion into the same tensors (an earlier
// FPC_FLAG_ASYNC_DENSE call) must finish first.
template <class G, class F>
static int launch_incremental(ObserveParams p, DenseOut d, const DeviceState &S, cudaStream_t st, F after_rules) {
  if (S.last >= 0 && S.last_async) CK(cudaStreamWaitEvent(st, S.expand_done[S.last], 0));
  const Records &r = d.track->rec;
  p.cells = d.planes ? r.cells[r.cur_cells] : nullptr;
  p.flats = d.mask ? r.flats[r.cur_flats] : nullptr;
  p.inc_planes = d.planes;
  p.inc_mask = d.mask;
  rules_kernel<G><<<(p.n + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK, BLOCK_THREADS, 0, st>>>(p);
  CK(cudaGetLastError());
  return after_rules();
}

// Is the caller running ahead of the device (both internal streams still have work queued), or does this call find
// one of them idle -- a run of dense calls starting up, or a host that waits for every step's results?  Asked before
// the call enqueues anything; never during stream capture, where querying a stream is not allowed (a captured call
// counts as running ahead).
static bool finds_stream_idle(const DeviceState &S, cudaStream_t st) {
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) cudaGetLastError(), cap = cudaStreamCaptureStatusActive;
  if (cap != cudaStreamCaptureStatusNone) return false;
  const bool idle = cudaStreamQuery(S.side) == cudaSuccess || cudaStreamQuery(S.hi) == cudaSuccess;
  cudaGetLastError();  // "not ready" is reported through the error state
  return idle;
}

// Which event marks the end of the expansion in slot b.  A TIMESTAMPED record is the robust one: measured on B200
// (tools/overlap_probe.py, DESIGN.md section 3 item 5) it costs ~2 us per step against a plain record when the caller
// runs far ahead of the device (76.3 vs 74.2 us per step), but with the plain record a loop that starts from
// an idle device loses ~250 us (20 steps: ~90 vs 79 us per step), and a caller that waits for every step's results
// before issuing the next one falls into a mode of 176 us per step (83 us with the timestamped record).  So: the
// timestamped record whenever a call finds an internal stream idle, and for the STARTUP_CALLS calls after that; the
// plain one only while the caller keeps both streams busy.
static cudaEvent_t end_event(DeviceState &S, int b, bool found_idle) {
  constexpr int STARTUP_CALLS = 8;
  if (found_idle) S.startup_left = STARTUP_CALLS;
  S.expand_done[b] = S.startup_left > 0 ? S.expand_done_stamped[b] : S.expand_done_plain[b];
  if (S.startup_left > 0) --S.startup_left;
  return S.expand_done[b];
}

// Full rewrite: rules_kernel on the high-priority stream forked from the caller's, expand_kernel on the side stream
// once the records exist; unless FPC_FLAG_ASYNC_DENSE is set the caller's stream then waits for the expansion.
template <class G, class F>
static int launch_full(ObserveParams p, DenseOut d, DeviceState &S, cudaStream_t st, F after_rules) {
  const bool found_idle = finds_stream_idle(S, st);
  const int b = S.parity;
  S.parity ^= 1;
  // growing the handle-less records (a handle's fit its batch): earlier launches may still use the old ones
  Records &r = d.track ? d.track->rec : S.ws;
  if ((size_t)p.n > r.games) {
    CK(cudaStreamSynchronize(st));
    CK(cudaStreamSynchronize(S.side));
    CK(cudaStreamSynchronize(S.hi));
    int rc = r.reserve((size_t)p.n);
    if (rc != FPC_OK) return rc;
  }
  if (d.planes) r.cur_cells ^= 1, p.cells = r.cells[r.cur_cells];
  if (d.mask) r.cur_flats ^= 1, p.flats = r.flats[r.cur_flats];
  CK(cudaEventRecord(S.fork, st));
  CK(cudaStreamWaitEvent(S.hi, S.fork, 0));
  // The half of the records this call writes was last read by an expansion at least two full rewrites earlier on this
  // thread and device: each tensor's records alternate halves, and only full rewrites flip them.  All those expansions
  // run in order on the one side stream, so waiting for the expansion two calls back (slot b) covers it.  Incremental
  // calls read the records on the caller's stream, which the fork orders.
  if (S.expand_recorded[b]) CK(cudaStreamWaitEvent(S.hi, S.expand_done[b], 0));
  // Both kernels ask for the same shared-memory carveout: CTAs of rules_kernel (14 KB of shared memory each) and of
  // expand_kernel (none) share SMs, and an SM only changes its L1 / shared split when it is empty.
  if (!((S.carveout_set >> G::R) & 1u)) {
    CK(cudaFuncSetAttribute(rules_kernel<G>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    CK(cudaFuncSetAttribute(expand_kernel<G>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    S.carveout_set |= 1u << G::R;
  }
  LaunchTimes *t = S.prof_on && S.prof_n < PROF_MAX ? &S.prof[S.prof_n] : nullptr;
  if (t) CK(cudaEventRecord(t->rules[0], S.hi));
  rules_kernel<G><<<(p.n + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK, BLOCK_THREADS, 0, S.hi>>>(p);
  CK(cudaGetLastError());
  if (t) CK(cudaEventRecord(t->rules[1], S.hi));
  CK(cudaEventRecord(S.rules_done[b], S.hi));
  CK(cudaStreamWaitEvent(st, S.rules_done[b], 0));
  const int rc = after_rules();
  if (rc != FPC_OK) return rc;
  CK(cudaStreamWaitEvent(S.side, S.rules_done[b], 0));
  if (t) CK(cudaEventRecord(t->expand[0], S.side));
  expand_kernel<G><<<p.n < S.sms ? p.n : S.sms, EXPAND_THREADS, 0, S.side>>>(p.cells, d.planes, p.flats, d.mask, p.n);
  CK(cudaGetLastError());
  if (t) {
    CK(cudaEventRecord(t->expand[1], S.side));
    ++S.prof_n;
  }
  const cudaEvent_t done = end_event(S, b, found_idle);
  CK(cudaEventRecord(done, S.side));
  S.expand_recorded[b] = true;
  S.last = b;
  S.last_async = (d.flags & FPC_FLAG_ASYNC_DENSE) != 0;
  if (!S.last_async) CK(cudaStreamWaitEvent(st, done, 0));
  return FPC_OK;
}

// after_rules (may be a no-op) runs right after the rules kernel is enqueued: the host-buffer entry points start their
// device-to-host copies of the compact results there.
template <class G, class F>
static int launch_observe(ObserveParams p, DenseOut d, cudaStream_t st, F after_rules) {
  if (p.n == 0) return FPC_OK;
  if (!d.planes && !d.mask) {  // rules only: one launch on the caller's stream
    rules_kernel<G><<<(p.n + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK, BLOCK_THREADS, 0, st>>>(p);
    CK(cudaGetLastError());
    return after_rules();
  }
  if ((reinterpret_cast<uintptr_t>(d.planes) | reinterpret_cast<uintptr_t>(d.mask)) & 15)
    return fail(FPC_ERR_ARG, "planes / mask must be 16-byte aligned");
  DeviceState *S = nullptr;
  int rc = device_state(&S, true);
  if (rc != FPC_OK) return rc;
  fpc_dense_track *T = d.track;
  if (T) {
    if (T->magic != TRACK_MAGIC) return fail(FPC_ERR_ARG, "fpc_dense_track: not a live handle");
    if (T->device != S->device || T->R != G::R || T->n != p.n) return fail(FPC_ERR_ARG, "fpc_dense_track: made for another device / board size / batch");
    // a handle follows one planes tensor and one mask tensor; being used with another one starts over for that tensor
    if (d.planes && d.planes != T->planes) T->planes = d.planes, T->known_planes = false;
    if (d.mask && d.mask != T->mask) T->mask = d.mask, T->known_mask = false;
    if ((d.flags & FPC_FLAG_INCREMENTAL) && (!d.planes || T->known_planes) && (!d.mask || T->known_mask))
      return launch_incremental<G>(p, d, *S, st, after_rules);
    // the full rewrite leaves each tensor it writes holding exactly its new record
    if (d.planes) T->known_planes = true;
    if (d.mask) T->known_mask = true;
  }
  return launch_full<G>(p, d, *S, st, after_rules);
}
template <class G>
static int launch_make(const uint8_t *in, const uint64_t *moves, const int32_t *flat, int n, uint8_t *out,
                       int32_t *err, cudaStream_t st) {
  if (n == 0) return FPC_OK;
  const int blocks = (n + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
  make_kernel<G><<<blocks, WARPS_PER_BLOCK * 32, 0, st>>>(in, moves, flat, n, out, err);
  return cuda_check(cudaGetLastError(), "make_kernel launch");
}
template <class G>
static int launch_heuristic(const uint8_t *in, int n, int32_t *v, cudaStream_t st) {
  if (n == 0) return FPC_OK;
  const int blocks = (n + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
  heuristic_kernel<G><<<blocks, WARPS_PER_BLOCK * 32, 0, st>>>(in, n, v);
  return cuda_check(cudaGetLastError(), "heuristic_kernel launch");
}

// Viewer queries (src/cpp/board.cpp:120-232), one thread per (board, square): bits 0..3 IsAttackedByPlayer per colour,
// bits 4..5 chess::Board::IsAttackedByTeam per team.  Plain loops over the record's piece bytes: this is the pygame
// viewer's query, a few boards per call.
template <class G>
__global__ void __launch_bounds__(256) attack_map_kernel(const uint8_t *boards, int n, uint8_t *out) {
  constexpr int R = G::R;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * G::NSQ) return;
  const int g = idx / G::NSQ, sq = idx - g * G::NSQ;
  const uint8_t *b = boards + (size_t)g * G::REC;
  const int r0 = sq / R, c0 = sq - r0 * R;
  auto inb = [](int r, int c) { return r >= 0 && r < R && c >= 0 && c < R; };
  uint32_t bits = 0;
  // ---- IsAttackedByPlayer (src/cpp/board.cpp:142-209): "legal" there means inside the R x R index range only --------
  for (int d = 0; d < 8; ++d) {
    const int dr = (int)(int8_t)((0xFF'FF'01'01'00'FF'00'01ull >> (8 * d)) & 0xff);  // (1,0)(0,1)(-1,0)(0,-1)(1,1)(1,-1)(-1,1)(-1,-1)
    const int dc = (int)(int8_t)((0xFF'01'FF'01'FF'00'01'00ull >> (8 * d)) & 0xff);
    // pawns and kings on the eight neighbours
    if (inb(r0 + dr, c0 + dc)) {
      const uint32_t p = b[(r0 + dr) * R + c0 + dc];
      const int col = color_of(p), t = type_of(p);
      if (t == 5) bits |= 1u << col;  // KING (an empty square has type NO_PIECE)
      if (t == 0) {
        // PawnAttacks(pawn at (r0+dr, c0+dc), colour, target): row_diff = -dr, col_diff = -dc (engine/board.cpp:583-604)
        const int rd = -dr, cd = -dc;
        const bool a = col == 0 ? (rd == -1 && (cd == 1 || cd == -1)) : col == 1 ? (cd == 1 && (rd == 1 || rd == -1))
                     : col == 2 ? (rd == 1 && (cd == 1 || cd == -1)) : (cd == -1 && (rd == 1 || rd == -1));
        if (a) bits |= 1u << col;
      }
    }
    // sliders: the first piece on the ray decides, for its own colour only
    for (int r = r0 + dr, c = c0 + dc; inb(r, c); r += dr, c += dc) {
      const uint32_t p = b[r * R + c];
      if (!present(p)) continue;
      const int t = type_of(p);
      const bool diag = dr != 0 && dc != 0;
      if (t == 4 || (t == 2 && diag) || (t == 3 && !diag)) bits |= 1u << color_of(p);
      break;
    }
  }
  for (int k = 0; k < 8; ++k) {
    const int r = r0 + kdrow(k), c = c0 + kdcol(k);
    if (inb(r, c)) {
      const uint32_t p = b[r * R + c];
      if (type_of(p) == 1 && present(p)) bits |= 1u << color_of(p);
    }
  }
  // ---- IsAttackedByTeam (engine/board.cpp:606-786) ---------------------------------------------------------------
  for (int d = 0; d < 8; ++d) {
    const int dr = (int)(int8_t)((0xFF'FF'01'01'00'FF'00'01ull >> (8 * d)) & 0xff);
    const int dc = (int)(int8_t)((0xFF'01'FF'01'FF'00'01'00ull >> (8 * d)) & 0xff);
    const bool diag = dr != 0 && dc != 0;
    // rook rays are bounded by the index range, bishop rays by IsLegalLocation
    for (int r = r0 + dr, c = c0 + dc; diag ? (inb(r, c) && G::legal(r, c)) : inb(r, c); r += dr, c += dc) {
      const uint32_t p = b[r * R + c];
      if (!present(p)) continue;
      const int t = type_of(p);
      if (t == 4 || (t == 2 && diag) || (t == 3 && !diag)) bits |= 16u << team_of(p);
      break;
    }
    const int r = r0 + dr, c = c0 + dc;
    if (inb(r, c)) {
      const uint32_t p = b[r * R + c];
      if (present(p)) {
        const int col = color_of(p), t = type_of(p);
        if (t == 5 && G::legal(r, c)) bits |= 16u << team_of(p);
        if (t == 0 && diag) {
          // pos_row = (dr == 1), pos_col = (dc == 1): RED attacks from below, BLUE from the left, ...
          const bool a = col == 0 ? dr == 1 : col == 1 ? dc == -1 : col == 2 ? dr == -1 : dc == 1;
          if (a) bits |= 16u << team_of(p);
        }
      }
    }
  }
  for (int k = 0; k < 8; ++k) {
    const int r = r0 + kdrow(k), c = c0 + kdcol(k);
    if (inb(r, c) && G::legal(r, c)) {
      const uint32_t p = b[r * R + c];
      if (present(p) && type_of(p) == 1) bits |= 16u << team_of(p);
    }
  }
  out[idx] = (uint8_t)bits;
}
template <class G>
static int launch_attack_maps(const uint8_t *in, int n, uint8_t *out, cudaStream_t st) {
  if (n == 0) return FPC_OK;
  const int total = n * G::NSQ;
  attack_map_kernel<G><<<(total + 255) / 256, 256, 0, st>>>(in, n, out);
  return cuda_check(cudaGetLastError(), "attack_map_kernel launch");
}

template <class F>
static int do_observe(int R, const ObserveParams &p, DenseOut d, cudaStream_t st, F after_rules) {
  return dispatch(R, [&](auto g) { return launch_observe<decltype(g)>(p, d, st, after_rules); });
}
static int do_observe(int R, const ObserveParams &p, DenseOut d, cudaStream_t st) {
  return do_observe(R, p, d, st, [] { return FPC_OK; });
}
static int do_make(int R, const uint8_t *in, const uint64_t *moves, const int32_t *flat, int n, uint8_t *out,
                   int32_t *err, cudaStream_t st) {
  return dispatch(R, [&](auto g) { return launch_make<decltype(g)>(in, moves, flat, n, out, err, st); });
}
static int do_heuristic(int R, const uint8_t *in, int n, int32_t *v, cudaStream_t st) {
  return dispatch(R, [&](auto g) { return launch_heuristic<decltype(g)>(in, n, v, st); });
}
static int do_attack_maps(int R, const uint8_t *in, int n, uint8_t *out, cudaStream_t st) {
  return dispatch(R, [&](auto g) { return launch_attack_maps<decltype(g)>(in, n, out, st); });
}

}  // namespace fpc

using namespace fpc;

extern "C" {

const char *fpc_last_error(void) { return g_err.c_str(); }
int fpc_version(void) { return 100; }
int fpc_supported(int R) { return ia_of(R) > 0; }
int fpc_invalid_area(int R) { return ia_of(R); }
int fpc_record_bytes(int R) { return fpc_supported(R) ? ((R * R + 12 + 15) / 16) * 16 : FPC_ERR_ARG; }
int fpc_num_action_channels(int R) { return fpc_supported(R) ? 8 * R + 8 : FPC_ERR_ARG; }
int fpc_action_space_size(int R) { return fpc_supported(R) ? (8 * R + 8) * R * R : FPC_ERR_ARG; }
int fpc_state_space_size(int R) { return fpc_supported(R) ? 24 * R * R : FPC_ERR_ARG; }

static const int kQd[8][2] = {{0, -1}, {-1, -1}, {-1, 0}, {-1, 1}, {0, 1}, {1, 1}, {1, 0}, {1, -1}};   // move.cpp:13-14
static const int kKd[8][2] = {{-2, -1}, {-2, 1}, {-1, -2}, {-1, 2}, {1, -2}, {1, 2}, {2, -1}, {2, 1}}; // move.cpp:15-16

uint64_t fpc_move_from_flat(int R, int flat) {
  const int nsq = R * R;
  if (!fpc_supported(R) || flat < 0 || flat >= (8 * R + 8) * nsq) {
    fail(FPC_ERR_ARG, "flat index out of range");
    return ~0ull;
  }
  const int type = flat / nsq, pos = flat % nsq, row = pos / R, col = pos % R;
  int dr, dc;
  if (type < 8 * (R - 1)) {
    const int dir = type / (R - 1), dist = type % (R - 1) + 1;
    dc = kQd[dir][0] * dist;
    dr = kQd[dir][1] * dist;
  } else {
    int k = type - 8 * (R - 1);
    if (k > 7) k = 7;
    dc = kKd[k][0];
    dr = kKd[k][1];
  }
  const int tr = row + dr, tc = col + dc;
  const uint64_t to = (tr < 0 || tr >= R || tc < 0 || tc >= R) ? nsq : tr * R + tc;
  return (uint64_t)pos | (to << 8) | (0x18ull << 16) | (6ull << 24) | ((uint64_t)nsq << 32) | ((uint64_t)nsq << 40);
}

int fpc_move_flat_index(int R, uint64_t move) {
  if (!fpc_supported(R)) return fail(FPC_ERR_ARG, "unsupported board size");
  const int from = (int)(move & 0xff), to = (int)((move >> 8) & 0xff);
  // BoardLocation::GetRow/GetCol (engine/board.h:203-204) also decode the "missing" value R*R
  const int dx = to % R - from % R, dy = to / R - from / R;
  int plane = -1;
  for (int i = 0; i < 8 && plane < 0; ++i)
    for (int d = 1; d <= R - 1; ++d)
      if (dx == kQd[i][0] * d && dy == kQd[i][1] * d) { plane = i * (R - 1) + d - 1; break; }
  for (int i = 0; i < 8 && plane < 0; ++i)
    if (dx == kKd[i][0] && dy == kKd[i][1]) plane = 8 * (R - 1) + i;
  if (plane < 0) return -1;
  return plane * R * R + (from / R) * R + from % R;
}

int fpc_record_from_fen(int R, const char *fen, int honour_castling, uint8_t *h_record) {
  if (!fpc_supported(R) || !fen || !h_record) return fail(FPC_ERR_ARG, "fpc_record_from_fen: bad argument");
  const int nsq = R * R, rec = fpc_record_bytes(R);
  std::string text;
  for (const char *c = fen; *c; ++c)
    if (*c != '\n' && *c != '\r' && *c != ' ') text += *c;
  auto split = [](const std::string &str, char sep) {
    std::vector<std::string> out;
    size_t at = 0;
    for (;;) {
      const size_t next = str.find(sep, at);
      out.push_back(str.substr(at, next == std::string::npos ? std::string::npos : next - at));
      if (next == std::string::npos) break;
      at = next + 1;
    }
    return out;
  };
  const std::vector<std::string> parts = split(text, '-');
  if (parts.size() < 5) return fail(FPC_ERR_ARG, "FEN string has too few fields");
  static const char turns[] = "RBYG";
  const char *tp = parts[0].size() == 1 ? strchr(turns, parts[0][0]) : nullptr;
  if (!tp || !*tp) return fail(FPC_ERR_ARG, "Invalid player character in FEN string");
  memset(h_record, 0, rec);
  memset(h_record, 0x18, nsq);
  h_record[nsq] = (uint8_t)(tp - turns);
  for (int c = 0; c < 4; ++c) h_record[nsq + 1 + c] = 0x80, h_record[nsq + 5 + c] = (uint8_t)nsq;
  const std::vector<std::string> ks = split(parts[2], ','), qs = split(parts[3], ',');
  if (ks.size() != 4) return fail(FPC_ERR_ARG, "Invalid kingside castling availability in FEN string");
  if (qs.size() != 4) return fail(FPC_ERR_ARG, "Invalid queenside castling availability in FEN string");
  if (honour_castling)
    for (int c = 0; c < 4; ++c) h_record[nsq + 1 + c] = (uint8_t)(0x80 | ((ks[c] == "1") << 6) | ((qs[c] == "1") << 5));
  const std::vector<std::string> rows = split(parts.back(), '/');
  if ((int)rows.size() > R) return fail(FPC_ERR_ARG, "Too many rows in piece placement");
  static const char colors[] = "rbyg", types[] = "PNBRQK";
  for (int row = 0; row < (int)rows.size(); ++row) {
    int col = 0;
    for (const std::string &cell : split(rows[row], ',')) {
      if (cell.empty()) return fail(FPC_ERR_ARG, "Empty column string in piece placement");
      const char *cp = strchr(colors, cell[0]);
      if (cp && *cp) {
        const char *ty = cell.size() == 2 ? strchr(types, cell[1]) : nullptr;
        if (!ty || !*ty) return fail(FPC_ERR_ARG, "Piece placement string for player must be of length 2");
        if (col >= R) return fail(FPC_ERR_ARG, "Piece placement outside the board");
        const int color = (int)(cp - colors), type = (int)(ty - types);
        h_record[row * R + col] = (uint8_t)(0x80 | (color << 5) | (type << 2));
        if (type == 5) h_record[nsq + 5 + color] = (uint8_t)(row * R + col);
        ++col;
      } else if (cell == "x") {
        ++col;
      } else {
        char *end = nullptr;
        const long n = strtol(cell.c_str(), &end, 10);
        if (!end || *end || n <= 0) return fail(FPC_ERR_ARG, "Invalid number of empty spaces in piece placement");
        col += (int)n;
      }
    }
  }
  return FPC_OK;
}

int fpc_profile_enable(int on) {
  DeviceState *S = nullptr;
  int rc = device_state(&S, true);
  if (rc != FPC_OK) return rc;
  if (on && S->prof.empty()) {
    S->prof.resize(PROF_MAX);
    for (LaunchTimes &t : S->prof)
      for (int i = 0; i < 2; ++i) {
        CK(cudaEventCreate(&t.rules[i]));
        CK(cudaEventCreate(&t.expand[i]));
      }
  }
  S->prof_on = on != 0;
  S->prof_n = 0;
  return FPC_OK;
}

int fpc_profile_read(int *launches, double *expand_ms, double *rules_ms) {
  DeviceState *S = nullptr;
  int rc = device_state(&S, true);
  if (rc != FPC_OK) return rc;
  CK(cudaStreamSynchronize(S->side));
  CK(cudaStreamSynchronize(S->hi));
  double total = 0, total_r = 0;
  for (int i = 0; i < S->prof_n; ++i) {
    const LaunchTimes &t = S->prof[i];
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, t.expand[0], t.expand[1]));
    total += ms;
    CK(cudaEventElapsedTime(&ms, t.rules[0], t.rules[1]));
    total_r += ms;
  }
  if (launches) *launches = S->prof_n;
  if (expand_ms) *expand_ms = total;
  if (rules_ms) *rules_ms = total_r;
  return FPC_OK;
}

int fpc_join(void *stream) {
  DeviceState *S = nullptr;
  int rc = device_state(&S, false);
  if (rc != FPC_OK) return rc;
  if (S->last >= 0) CK(cudaStreamWaitEvent((cudaStream_t)stream, S->expand_done[S->last], 0));
  return FPC_OK;
}

// Releases everything this host thread holds on the current device.
int fpc_shutdown(void) {
  DeviceState *S = nullptr;
  int rc = device_state(&S, false);
  if (rc != FPC_OK) return rc;
  if (S->side) {
    CK(cudaStreamSynchronize(S->side));
    CK(cudaStreamSynchronize(S->hi));
    cudaStreamDestroy(S->side);
    cudaStreamDestroy(S->hi);
    cudaEventDestroy(S->fork);
    for (int i = 0; i < 2; ++i) {
      cudaEventDestroy(S->rules_done[i]);
      cudaEventDestroy(S->expand_done_plain[i]);
      cudaEventDestroy(S->expand_done_stamped[i]);
    }
  }
  S->ws.release();
  for (LaunchTimes &t : S->prof)
    for (int i = 0; i < 2; ++i) cudaEventDestroy(t.rules[i]), cudaEventDestroy(t.expand[i]);
  *S = DeviceState();
  return FPC_OK;
}

fpc_dense_track *fpc_dense_track_create(int R, int n) {
  if (!fpc_supported(R) || n <= 0) {
    fail(FPC_ERR_ARG, "fpc_dense_track_create: bad argument");
    return nullptr;
  }
  int dev = 0;
  if (cuda_check(cudaGetDevice(&dev), "cudaGetDevice") != FPC_OK) return nullptr;
  fpc_dense_track *t = new fpc_dense_track();
  t->magic = TRACK_MAGIC;
  t->device = dev, t->R = R, t->n = n;
  t->planes = t->mask = nullptr;
  t->known_planes = t->known_mask = false;
  if (t->rec.reserve((size_t)n) != FPC_OK) {
    t->rec.release();
    delete t;
    return nullptr;
  }
  return t;
}

void fpc_dense_track_invalidate(fpc_dense_track *t) {
  if (t && t->magic == TRACK_MAGIC) t->known_planes = t->known_mask = false;
}

void fpc_dense_track_destroy(fpc_dense_track *t) {
  if (!t || t->magic != TRACK_MAGIC) return;
  int dev = 0;
  cudaGetDevice(&dev);
  cudaSetDevice(t->device);
  cudaDeviceSynchronize();  // kernels may still read the records
  t->rec.release();
  cudaSetDevice(dev);
  t->magic = 0;
  delete t;
}

int fpc_observe_tracked(fpc_dense_track *track, int R, const uint8_t *d_boards, int n, uint64_t *d_moves, int32_t *d_flat,
                        int32_t *d_counts, int32_t *d_status, float *d_planes, const int32_t *d_k, int k_all, float *d_mask,
                        int flags, void *stream) {
  if (n < 0 || (n > 0 && !d_boards)) return fail(FPC_ERR_ARG, "fpc_observe: bad boards/n");
  ObserveParams p{};
  p.boards_in = d_boards;
  p.n = n;
  p.need_movegen = (d_moves || d_flat || d_counts || d_status || d_mask) ? 1 : 0;
  p.moves = d_moves;
  p.flat = d_flat;
  p.counts = d_counts;
  p.status = d_status;
  p.k = d_k;
  p.k_all = k_all;
  return do_observe(R, p, DenseOut{d_planes, d_mask, flags, track}, (cudaStream_t)stream);
}

int fpc_observe(int R, const uint8_t *d_boards, int n, uint64_t *d_moves, int32_t *d_flat, int32_t *d_counts,
                int32_t *d_status, float *d_planes, const int32_t *d_k, int k_all, float *d_mask, int flags,
                void *stream) {
  return fpc_observe_tracked(nullptr, R, d_boards, n, d_moves, d_flat, d_counts, d_status, d_planes, d_k, k_all, d_mask,
                             flags, stream);
}

int fpc_encode(int R, const uint8_t *d_boards, int n, const int32_t *d_k, int k_all, float *d_planes, int flags,
               void *stream) {
  if (!d_planes && n > 0) return fail(FPC_ERR_ARG, "fpc_encode: null output");
  return fpc_observe(R, d_boards, n, nullptr, nullptr, nullptr, nullptr, d_planes, d_k, k_all, nullptr, flags,
                     stream);
}

int fpc_make_moves(int R, const uint8_t *d_in, const uint64_t *d_moves, int n, uint8_t *d_out, int32_t *d_err,
                   void *stream) {
  if (n < 0 || (n > 0 && (!d_in || !d_moves || !d_out))) return fail(FPC_ERR_ARG, "fpc_make_moves: bad argument");
  return do_make(R, d_in, d_moves, nullptr, n, d_out, d_err, (cudaStream_t)stream);
}

int fpc_make_index(int R, const uint8_t *d_in, const int32_t *d_flat, int n, uint8_t *d_out, int32_t *d_err,
                   void *stream) {
  if (n < 0 || (n > 0 && (!d_in || !d_flat || !d_out))) return fail(FPC_ERR_ARG, "fpc_make_index: bad argument");
  return do_make(R, d_in, nullptr, d_flat, n, d_out, d_err, (cudaStream_t)stream);
}

int fpc_heuristic(int R, const uint8_t *d_boards, int n, int32_t *d_value, void *stream) {
  if (n < 0 || (n > 0 && (!d_boards || !d_value))) return fail(FPC_ERR_ARG, "fpc_heuristic: bad argument");
  return do_heuristic(R, d_boards, n, d_value, (cudaStream_t)stream);
}

int fpc_attack_maps(int R, const uint8_t *d_boards, int n, uint8_t *d_out, void *stream) {
  if (n < 0 || (n > 0 && (!d_boards || !d_out))) return fail(FPC_ERR_ARG, "fpc_attack_maps: bad argument");
  return do_attack_maps(R, d_boards, n, d_out, (cudaStream_t)stream);
}

static int playout_params(ObserveParams &p, uint8_t *d_boards, int n, uint64_t seed, uint64_t *d_game, int32_t *d_ply,
                          const uint8_t *d_start, int max_plies, uint64_t game_stride, uint64_t *d_chosen,
                          int32_t *d_counts, int32_t *d_status, const int32_t *d_k, int k_all,
                          uint64_t *d_counters) {
  if (n < 0 || (n > 0 && (!d_boards || !d_game || !d_ply || !d_start)) || max_plies <= 0)
    return fail(FPC_ERR_ARG, "fpc_playout_step: bad argument");
  p = ObserveParams{};
  p.boards_in = d_boards;
  p.boards_out = d_boards;
  p.n = n;
  p.need_movegen = 1;
  p.counts = d_counts;
  p.status = d_status;
  p.k = d_k;
  p.k_all = k_all;
  p.playout = 1;
  p.seed = seed;
  p.game = d_game;
  p.ply = d_ply;
  p.start = d_start;
  p.max_plies = max_plies;
  p.game_stride = game_stride;
  p.chosen = d_chosen;
  p.counters = reinterpret_cast<unsigned long long *>(d_counters);
  return FPC_OK;
}

int fpc_playout_step_tracked(fpc_dense_track *track, int R, uint8_t *d_boards, int n, uint64_t seed, uint64_t *d_game,
                             int32_t *d_ply, const uint8_t *d_start, int max_plies, uint64_t game_stride, uint64_t *d_chosen,
                             int32_t *d_counts, int32_t *d_status, float *d_planes, const int32_t *d_k, int k_all,
                             float *d_mask, uint64_t *d_counters, int flags, void *stream) {
  ObserveParams p;
  int rc = playout_params(p, d_boards, n, seed, d_game, d_ply, d_start, max_plies, game_stride, d_chosen, d_counts,
                          d_status, d_k, k_all, d_counters);
  if (rc != FPC_OK) return rc;
  return do_observe(R, p, DenseOut{d_planes, d_mask, flags, track}, (cudaStream_t)stream);
}

int fpc_playout_step(int R, uint8_t *d_boards, int n, uint64_t seed, uint64_t *d_game, int32_t *d_ply,
                     const uint8_t *d_start, int max_plies, uint64_t game_stride, uint64_t *d_chosen,
                     int32_t *d_counts, int32_t *d_status, float *d_planes, const int32_t *d_k, int k_all,
                     float *d_mask, uint64_t *d_counters, int flags, void *stream) {
  return fpc_playout_step_tracked(nullptr, R, d_boards, n, seed, d_game, d_ply, d_start, max_plies, game_stride, d_chosen,
                                  d_counts, d_status, d_planes, d_k, k_all, d_mask, d_counters, flags, stream);
}

// ---- host-buffer context ---------------------------------------------------------------------

struct fpc_ctx {
  int device, R, max_n, rec;
  cudaStream_t stream, own_stream;  // stream = own_stream unless fpc_ctx_set_stream redirected the work
  uint8_t *d_boards, *d_boards2, *d_start;
  uint64_t *d_moves, *d_game;
  int32_t *d_flat, *d_counts, *d_status, *d_ply, *d_err;
  float *d_planes, *d_mask;   // lazily allocated for host-destination dense outputs
  uint8_t h_start_cache[256];
  bool start_valid;
};

fpc_ctx *fpc_ctx_create(int device, int R, int max_n) {
  if (!fpc_supported(R) || max_n <= 0) {
    fail(FPC_ERR_ARG, "fpc_ctx_create: bad argument");
    return nullptr;
  }
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0 || device < 0 || device >= count) {
    fail(FPC_ERR_CUDA, "fpc_ctx_create: no usable CUDA device (there is no CPU fallback)");
    return nullptr;
  }
  if (cuda_check(cudaSetDevice(device), "cudaSetDevice") != FPC_OK) return nullptr;
  fpc_ctx *c = new fpc_ctx();
  memset(c, 0, sizeof *c);
  c->device = device;
  c->R = R;
  c->max_n = max_n;
  c->rec = fpc_record_bytes(R);
  const size_t n = (size_t)max_n;
  bool ok = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) == cudaSuccess;
  c->stream = c->own_stream;
  ok = ok && cudaMalloc(&c->d_boards, n * c->rec) == cudaSuccess;
  ok = ok && cudaMalloc(&c->d_boards2, n * c->rec) == cudaSuccess;
  ok = ok && cudaMalloc(&c->d_start, c->rec) == cudaSuccess;
  ok = ok && cudaMalloc(&c->d_moves, n * FPC_MAX_MOVES * sizeof(uint64_t)) == cudaSuccess;
  ok = ok && cudaMalloc(&c->d_flat, n * FPC_MAX_MOVES * sizeof(int32_t)) == cudaSuccess;
  ok = ok && cudaMalloc(&c->d_game, n * sizeof(uint64_t)) == cudaSuccess;
  ok = ok && cudaMalloc(&c->d_counts, n * sizeof(int32_t)) == cudaSuccess;
  ok = ok && cudaMalloc(&c->d_status, n * sizeof(int32_t)) == cudaSuccess;
  ok = ok && cudaMalloc(&c->d_ply, n * sizeof(int32_t)) == cudaSuccess;
  ok = ok && cudaMalloc(&c->d_err, n * sizeof(int32_t)) == cudaSuccess;
  if (!ok) {
    fail(FPC_ERR_CUDA, std::string("fpc_ctx_create: ") + cudaGetErrorString(cudaGetLastError()));
    fpc_ctx_destroy(c);
    return nullptr;
  }
  return c;
}

void fpc_ctx_destroy(fpc_ctx *c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  cudaFree(c->d_boards);
  cudaFree(c->d_boards2);
  cudaFree(c->d_start);
  cudaFree(c->d_moves);
  cudaFree(c->d_flat);
  cudaFree(c->d_game);
  cudaFree(c->d_counts);
  cudaFree(c->d_status);
  cudaFree(c->d_ply);
  cudaFree(c->d_err);
  cudaFree(c->d_planes);
  cudaFree(c->d_mask);
  delete c;
}

void *fpc_ctx_stream(fpc_ctx *c) { return c ? (void *)c->stream : nullptr; }


// The host-buffer calls run on the context's device and leave the caller's current device as they found it.
struct DevGuard {
  int prev = -1;
  bool switched = false;
  int enter(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev == dev) return FPC_OK;
    int rc = cuda_check(cudaSetDevice(dev), "cudaSetDevice");
    switched = rc == FPC_OK && prev >= 0;
    return rc;
  }
  ~DevGuard() {
    if (switched) cudaSetDevice(prev);
  }
};
static int ctx_check(fpc_ctx *c, int n, const char *who, DevGuard &guard) {
  if (!c) return fail(FPC_ERR_ARG, std::string(who) + ": null context");
  if (n < 0 || n > c->max_n) return fail(FPC_ERR_ARG, std::string(who) + ": n exceeds the context capacity");
  return guard.enter(c->device);
}

int fpc_ctx_sync(fpc_ctx *c) {
  DevGuard guard_;
  int rc = ctx_check(c, 0, "fpc_ctx_sync", guard_);
  if (rc != FPC_OK) return rc;
  rc = fpc_join(c->stream);
  if (rc != FPC_OK) return rc;
  return cuda_check(cudaStreamSynchronize(c->stream), "cudaStreamSynchronize");
}

int fpc_host_observe(fpc_ctx *c, const uint8_t *h_boards, int n, uint64_t *h_moves, int32_t *h_flat,
                     int32_t *h_counts, int32_t *h_status, float *h_planes, float *d_planes, int k_all,
                     float *h_mask, float *d_mask) {
  DevGuard guard_;
  int rc = ctx_check(c, n, "fpc_host_observe", guard_);
  if (rc != FPC_OK) return rc;
  if (n == 0) return FPC_OK;
  if (!h_boards) return fail(FPC_ERR_ARG, "fpc_host_observe: null boards");
  const size_t N = (size_t)n;
  const size_t ssz = (size_t)fpc_state_space_size(c->R), asz = (size_t)fpc_action_space_size(c->R);
  if (h_planes && !d_planes) {
    if (!c->d_planes) CK(cudaMalloc(&c->d_planes, (size_t)c->max_n * ssz * sizeof(float)));
    d_planes = c->d_planes;
  }
  if (h_mask && !d_mask) {
    if (!c->d_mask) CK(cudaMalloc(&c->d_mask, (size_t)c->max_n * asz * sizeof(float)));
    d_mask = c->d_mask;
  }
  CK(cudaMemcpyAsync(c->d_boards, h_boards, N * c->rec, cudaMemcpyHostToDevice, c->stream));
  rc = fpc_observe(c->R, c->d_boards, n, h_moves ? c->d_moves : nullptr, h_flat ? c->d_flat : nullptr,
                   (h_counts || h_moves || h_flat) ? c->d_counts : nullptr, h_status ? c->d_status : nullptr,
                   d_planes, nullptr, k_all, d_mask, 0, c->stream);
  if (rc != FPC_OK) return rc;
  if (h_counts) CK(cudaMemcpyAsync(h_counts, c->d_counts, N * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  if (h_status) CK(cudaMemcpyAsync(h_status, c->d_status, N * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  if (h_moves)
    CK(cudaMemcpyAsync(h_moves, c->d_moves, N * FPC_MAX_MOVES * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
  if (h_flat)
    CK(cudaMemcpyAsync(h_flat, c->d_flat, N * FPC_MAX_MOVES * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  if (h_planes) CK(cudaMemcpyAsync(h_planes, d_planes, N * ssz * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  if (h_mask) CK(cudaMemcpyAsync(h_mask, d_mask, N * asz * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return FPC_OK;
}

static int host_make(fpc_ctx *c, const uint8_t *h_in, const uint64_t *h_moves, const int32_t *h_flat, int n,
                     uint8_t *h_out, int32_t *h_err) {
  DevGuard guard_;
  int rc = ctx_check(c, n, "fpc_host_make", guard_);
  if (rc != FPC_OK) return rc;
  if (n == 0) return FPC_OK;
  if (!h_in || !h_out || (!h_moves && !h_flat)) return fail(FPC_ERR_ARG, "fpc_host_make: null argument");
  const size_t N = (size_t)n;
  CK(cudaMemcpyAsync(c->d_boards, h_in, N * c->rec, cudaMemcpyHostToDevice, c->stream));
  if (h_moves) {
    CK(cudaMemcpyAsync(c->d_moves, h_moves, N * sizeof(uint64_t), cudaMemcpyHostToDevice, c->stream));
    rc = fpc_make_moves(c->R, c->d_boards, c->d_moves, n, c->d_boards2, c->d_err, c->stream);
  } else {
    CK(cudaMemcpyAsync(c->d_flat, h_flat, N * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
    rc = fpc_make_index(c->R, c->d_boards, c->d_flat, n, c->d_boards2, c->d_err, c->stream);
  }
  if (rc != FPC_OK) return rc;
  CK(cudaMemcpyAsync(h_out, c->d_boards2, N * c->rec, cudaMemcpyDeviceToHost, c->stream));
  if (h_err) CK(cudaMemcpyAsync(h_err, c->d_err, N * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return FPC_OK;
}

int fpc_host_make_moves(fpc_ctx *c, const uint8_t *h_in, const uint64_t *h_moves, int n, uint8_t *h_out,
                        int32_t *h_err) {
  return host_make(c, h_in, h_moves, nullptr, n, h_out, h_err);
}
int fpc_host_make_index(fpc_ctx *c, const uint8_t *h_in, const int32_t *h_flat, int n, uint8_t *h_out,
                        int32_t *h_err) {
  return host_make(c, h_in, nullptr, h_flat, n, h_out, h_err);
}

// Device alias of a pinned (page-locked, mapped) host pointer, or null for pageable memory.
static void *mapped_alias(const void *h) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, h) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return a.type == cudaMemoryTypeHost ? a.devicePointer : nullptr;
}

int fpc_host_playout_step(fpc_ctx *c, uint8_t *h_boards, int n, uint64_t seed, uint64_t *h_game, int32_t *h_ply,
                          const uint8_t *h_start, int max_plies, uint64_t game_stride, int32_t *h_counts,
                          int32_t *h_status, float *d_planes, int k_all, float *d_mask, int flags) {
  DevGuard guard_;
  int rc = ctx_check(c, n, "fpc_host_playout_step", guard_);
  if (rc != FPC_OK) return rc;
  if (n == 0) return FPC_OK;
  if (!h_boards || !h_game || !h_ply || !h_start) return fail(FPC_ERR_ARG, "fpc_host_playout_step: null argument");
  const size_t N = (size_t)n;
  // the start record only changes between runs: upload it when it differs from the cached copy
  if (!c->start_valid || memcmp(c->h_start_cache, h_start, c->rec) != 0) {
    memcpy(c->h_start_cache, h_start, c->rec);
    CK(cudaMemcpyAsync(c->d_start, c->h_start_cache, c->rec, cudaMemcpyHostToDevice, c->stream));
    c->start_valid = true;
  }
  ObserveParams p;
  // Zero-copy: when every host buffer is pinned, the rules kernel reads the records straight from
  // host memory and writes its results straight back over PCIe -- no staging copies, one launch.
  uint8_t *m_boards = (uint8_t *)mapped_alias(h_boards);
  uint64_t *m_game = (uint64_t *)mapped_alias(h_game);
  int32_t *m_ply = (int32_t *)mapped_alias(h_ply);
  int32_t *m_counts = h_counts ? (int32_t *)mapped_alias(h_counts) : nullptr;
  int32_t *m_status = h_status ? (int32_t *)mapped_alias(h_status) : nullptr;
  if (m_boards && m_game && m_ply && (!h_counts || m_counts) && (!h_status || m_status)) {
    rc = playout_params(p, m_boards, n, seed, m_game, m_ply, c->d_start, max_plies, game_stride, nullptr, m_counts,
                        m_status, nullptr, k_all, nullptr);
    if (rc != FPC_OK) return rc;
    rc = do_observe(c->R, p, DenseOut{d_planes, d_mask, flags, nullptr}, c->stream);
    if (rc != FPC_OK) return rc;
    CK(cudaStreamSynchronize(c->stream));
    return FPC_OK;
  }
  CK(cudaMemcpyAsync(c->d_boards, h_boards, N * c->rec, cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemcpyAsync(c->d_game, h_game, N * sizeof(uint64_t), cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemcpyAsync(c->d_ply, h_ply, N * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
  rc = playout_params(p, c->d_boards, n, seed, c->d_game, c->d_ply, c->d_start, max_plies, game_stride, nullptr,
                      c->d_counts, c->d_status, nullptr, k_all, nullptr);
  if (rc != FPC_OK) return rc;
  // the compact results go back to the host while the dense outputs are still being written
  rc = do_observe(c->R, p, DenseOut{d_planes, d_mask, flags, nullptr}, c->stream, [&]() -> int {
    CK(cudaMemcpyAsync(h_boards, c->d_boards, N * c->rec, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_game, c->d_game, N * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_ply, c->d_ply, N * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    if (h_counts) CK(cudaMemcpyAsync(h_counts, c->d_counts, N * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    if (h_status) CK(cudaMemcpyAsync(h_status, c->d_status, N * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    return FPC_OK;
  });
  if (rc != FPC_OK) return rc;
  CK(cudaStreamSynchronize(c->stream));
  return FPC_OK;
}

int fpc_ctx_set_stream(fpc_ctx *c, void *stream) {
  if (!c) return fail(FPC_ERR_ARG, "fpc_ctx_set_stream: null context");
  c->stream = stream ? (cudaStream_t)stream : c->own_stream;
  return FPC_OK;
}

int fpc_current_device(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cudaGetLastError();
    return fail(FPC_ERR_CUDA, "fpc_current_device: no usable CUDA device (there is no CPU fallback)");
  }
  return dev;
}

void *fpc_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cuda_check(cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault), "cudaHostAlloc") != FPC_OK) return nullptr;
  return p;
}
void fpc_host_free(void *p) {
  if (p) cudaFreeHost(p);
}

int fpc_host_expand(fpc_ctx *c, const uint8_t *h_parents, const uint64_t *h_moves, int n, uint8_t *h_children,
                    int32_t *h_err, int32_t *h_counts, int32_t *h_status) {
  DevGuard guard_;
  int rc = ctx_check(c, n, "fpc_host_expand", guard_);
  if (rc != FPC_OK) return rc;
  if (n == 0) return FPC_OK;
  if (!h_parents || !h_moves || !h_children) return fail(FPC_ERR_ARG, "fpc_host_expand: null argument");
  const size_t N = (size_t)n;
  CK(cudaMemcpyAsync(c->d_boards, h_parents, N * c->rec, cudaMemcpyHostToDevice, c->stream));
  // the moves to make sit in the first n slots of the move buffer; the children's legal moves overwrite it afterwards
  CK(cudaMemcpyAsync(c->d_moves, h_moves, N * sizeof(uint64_t), cudaMemcpyHostToDevice, c->stream));
  rc = fpc_make_moves(c->R, c->d_boards, c->d_moves, n, c->d_boards2, c->d_err, c->stream);
  if (rc != FPC_OK) return rc;
  rc = fpc_observe(c->R, c->d_boards2, n, c->d_moves, nullptr, c->d_counts, c->d_status, nullptr, nullptr, -1, nullptr, 0,
                   c->stream);
  if (rc != FPC_OK) return rc;
  CK(cudaMemcpyAsync(h_children, c->d_boards2, N * c->rec, cudaMemcpyDeviceToHost, c->stream));
  if (h_err) CK(cudaMemcpyAsync(h_err, c->d_err, N * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  if (h_counts) CK(cudaMemcpyAsync(h_counts, c->d_counts, N * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  if (h_status) CK(cudaMemcpyAsync(h_status, c->d_status, N * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return FPC_OK;
}

int fpc_host_fetch_moves(fpc_ctx *c, int n, int stride, uint64_t *h_moves) {
  DevGuard guard_;
  int rc = ctx_check(c, n, "fpc_host_fetch_moves", guard_);
  if (rc != FPC_OK) return rc;
  if (n == 0 || stride == 0) return FPC_OK;
  if (!h_moves || stride < 0 || stride > FPC_MAX_MOVES) return fail(FPC_ERR_ARG, "fpc_host_fetch_moves: bad argument");
  CK(cudaMemcpy2DAsync(h_moves, (size_t)stride * sizeof(uint64_t), c->d_moves, (size_t)FPC_MAX_MOVES * sizeof(uint64_t),
                       (size_t)stride * sizeof(uint64_t), (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return FPC_OK;
}

int fpc_host_encode(fpc_ctx *c, const uint8_t *h_boards, int n, int k_all, float *d_planes) {
  DevGuard guard_;
  int rc = ctx_check(c, n, "fpc_host_encode", guard_);
  if (rc != FPC_OK) return rc;
  if (n == 0) return FPC_OK;
  if (!h_boards || !d_planes) return fail(FPC_ERR_ARG, "fpc_host_encode: null argument");
  CK(cudaMemcpyAsync(c->d_boards, h_boards, (size_t)n * c->rec, cudaMemcpyHostToDevice, c->stream));
  rc = fpc_encode(c->R, c->d_boards, n, nullptr, k_all, d_planes, 0, c->stream);
  if (rc != FPC_OK) return rc;
  CK(cudaStreamSynchronize(c->stream));  // the host buffer and d_boards are free again; the planes are complete
  return FPC_OK;
}

int fpc_host_heuristic(fpc_ctx *c, const uint8_t *h_boards, int n, int32_t *h_value) {
  DevGuard guard_;
  int rc = ctx_check(c, n, "fpc_host_heuristic", guard_);
  if (rc != FPC_OK) return rc;
  if (n == 0) return FPC_OK;
  if (!h_boards || !h_value) return fail(FPC_ERR_ARG, "fpc_host_heuristic: null argument");
  CK(cudaMemcpyAsync(c->d_boards, h_boards, (size_t)n * c->rec, cudaMemcpyHostToDevice, c->stream));
  rc = fpc_heuristic(c->R, c->d_boards, n, c->d_err, c->stream);
  if (rc != FPC_OK) return rc;
  CK(cudaMemcpyAsync(h_value, c->d_err, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return FPC_OK;
}

int fpc_host_attack_maps(fpc_ctx *c, const uint8_t *h_boards, int n, uint8_t *h_out) {
  DevGuard guard_;
  int rc = ctx_check(c, n, "fpc_host_attack_maps", guard_);
  if (rc != FPC_OK) return rc;
  if (n == 0) return FPC_OK;
  if (!h_boards || !h_out) return fail(FPC_ERR_ARG, "fpc_host_attack_maps: null argument");
  const size_t nsq = (size_t)c->R * c->R;
  uint8_t *d_out = reinterpret_cast<uint8_t *>(c->d_flat);  // [n][FPC_MAX_MOVES] int32 >= [n][R*R] bytes
  CK(cudaMemcpyAsync(c->d_boards, h_boards, (size_t)n * c->rec, cudaMemcpyHostToDevice, c->stream));
  rc = fpc_attack_maps(c->R, c->d_boards, n, d_out, c->stream);
  if (rc != FPC_OK) return rc;
  CK(cudaMemcpyAsync(h_out, d_out, (size_t)n * nsq, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return FPC_OK;
}

// ---- environment-owned store + DLPack -------------------------------------------------------------------------

struct fpc_env {
  uint32_t magic;
  int device, R, n, rec;
  long refs;  // 1 for the owner until fpc_env_destroy, +1 per exported DLManagedTensor
  cudaStream_t stream;
  uint8_t *boards, *start;
  uint64_t *moves, *game, *counters;
  int32_t *flat, *counts, *status, *ply;
  float *planes, *mask;
};
static constexpr uint32_t ENV_MAGIC = 0x46504345u;

static void env_release(fpc_env *e) {
  if (__atomic_sub_fetch(&e->refs, 1, __ATOMIC_ACQ_REL) != 0) return;
  int dev = 0;
  cudaGetDevice(&dev);
  cudaSetDevice(e->device);
  if (e->stream) {
    cudaStreamSynchronize(e->stream);
    cudaStreamDestroy(e->stream);
  }
  cudaFree(e->boards), cudaFree(e->start), cudaFree(e->moves), cudaFree(e->game), cudaFree(e->counters);
  cudaFree(e->flat), cudaFree(e->counts), cudaFree(e->status), cudaFree(e->ply), cudaFree(e->planes), cudaFree(e->mask);
  cudaSetDevice(dev);
  e->magic = 0;
  delete e;
}

static int env_check(fpc_env *e, const char *who, DevGuard &guard) {
  if (!e || e->magic != ENV_MAGIC) return fail(FPC_ERR_ARG, std::string(who) + ": not an environment");
  return guard.enter(e->device);
}

fpc_env *fpc_env_create(int device, int R, int n) {
  if (!fpc_supported(R) || n <= 0) {
    fail(FPC_ERR_ARG, "fpc_env_create: bad argument");
    return nullptr;
  }
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0 || device < 0 || device >= count) {
    cudaGetLastError();
    fail(FPC_ERR_CUDA, "fpc_env_create: no usable CUDA device (there is no CPU fallback)");
    return nullptr;
  }
  if (cuda_check(cudaSetDevice(device), "cudaSetDevice") != FPC_OK) return nullptr;
  fpc_env *e = new fpc_env();
  memset(e, 0, sizeof *e);
  e->magic = ENV_MAGIC, e->device = device, e->R = R, e->n = n, e->rec = fpc_record_bytes(R), e->refs = 1;
  const size_t N = (size_t)n;
  bool ok = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaMalloc(&e->boards, N * e->rec) == cudaSuccess && cudaMalloc(&e->start, e->rec) == cudaSuccess;
  ok = ok && cudaMalloc(&e->moves, N * FPC_MAX_MOVES * sizeof(uint64_t)) == cudaSuccess;
  ok = ok && cudaMalloc(&e->flat, N * FPC_MAX_MOVES * sizeof(int32_t)) == cudaSuccess;
  ok = ok && cudaMalloc(&e->game, N * sizeof(uint64_t)) == cudaSuccess && cudaMalloc(&e->counters, 8 * sizeof(uint64_t)) == cudaSuccess;
  ok = ok && cudaMalloc(&e->counts, N * sizeof(int32_t)) == cudaSuccess && cudaMalloc(&e->status, N * sizeof(int32_t)) == cudaSuccess;
  ok = ok && cudaMalloc(&e->ply, N * sizeof(int32_t)) == cudaSuccess;
  ok = ok && cudaMalloc(&e->planes, N * fpc_state_space_size(R) * sizeof(float)) == cudaSuccess;
  ok = ok && cudaMalloc(&e->mask, N * fpc_action_space_size(R) * sizeof(float)) == cudaSuccess;
  if (ok) {
    // game ids 0..n-1 (one id step per slot: game_stride = n re-seeds slot g with g + n, g + 2n, ...), ply 0
    std::vector<uint64_t> ids(N);
    for (size_t i = 0; i < N; ++i) ids[i] = i;
    ok = cudaMemcpyAsync(e->game, ids.data(), N * sizeof(uint64_t), cudaMemcpyHostToDevice, e->stream) == cudaSuccess;
    ok = ok && cudaMemsetAsync(e->ply, 0, N * sizeof(int32_t), e->stream) == cudaSuccess;
    ok = ok && cudaMemsetAsync(e->counters, 0, 8 * sizeof(uint64_t), e->stream) == cudaSuccess;
    ok = ok && cudaMemsetAsync(e->boards, 0, N * e->rec, e->stream) == cudaSuccess;
    ok = ok && cudaStreamSynchronize(e->stream) == cudaSuccess;
  }
  if (!ok) {
    fail(FPC_ERR_CUDA, std::string("fpc_env_create: ") + cudaGetErrorString(cudaGetLastError()));
    env_release(e);
    return nullptr;
  }
  return e;
}

void fpc_env_destroy(fpc_env *e) {
  if (e && e->magic == ENV_MAGIC) env_release(e);
}
void *fpc_env_stream(fpc_env *e) { return (e && e->magic == ENV_MAGIC) ? (void *)e->stream : nullptr; }
int fpc_env_sync(fpc_env *e) {
  DevGuard guard_;
  int rc = env_check(e, "fpc_env_sync", guard_);
  if (rc != FPC_OK) return rc;
  return cuda_check(cudaStreamSynchronize(e->stream), "cudaStreamSynchronize");
}

int fpc_env_set_boards(fpc_env *e, const uint8_t *h_boards, int first, int count) {
  DevGuard guard_;
  int rc = env_check(e, "fpc_env_set_boards", guard_);
  if (rc != FPC_OK) return rc;
  if (!h_boards || first < 0 || count < 0 || first + count > e->n) return fail(FPC_ERR_ARG, "fpc_env_set_boards: bad range");
  CK(cudaMemcpyAsync(e->boards + (size_t)first * e->rec, h_boards, (size_t)count * e->rec, cudaMemcpyHostToDevice, e->stream));
  CK(cudaMemsetAsync(e->ply + first, 0, (size_t)count * sizeof(int32_t), e->stream));
  return cuda_check(cudaStreamSynchronize(e->stream), "cudaStreamSynchronize");  // the host buffer is free again
}
int fpc_env_get_boards(fpc_env *e, uint8_t *h_boards, int first, int count) {
  DevGuard guard_;
  int rc = env_check(e, "fpc_env_get_boards", guard_);
  if (rc != FPC_OK) return rc;
  if (!h_boards || first < 0 || count < 0 || first + count > e->n) return fail(FPC_ERR_ARG, "fpc_env_get_boards: bad range");
  CK(cudaMemcpyAsync(h_boards, e->boards + (size_t)first * e->rec, (size_t)count * e->rec, cudaMemcpyDeviceToHost, e->stream));
  return cuda_check(cudaStreamSynchronize(e->stream), "cudaStreamSynchronize");
}

int fpc_env_observe(fpc_env *e, int which, int k_all) {
  DevGuard guard_;
  int rc = env_check(e, "fpc_env_observe", guard_);
  if (rc != FPC_OK) return rc;
  return fpc_observe(e->R, e->boards, e->n, (which & FPC_ENV_MOVES) ? e->moves : nullptr, (which & FPC_ENV_FLAT) ? e->flat : nullptr,
                     e->counts, e->status, (which & FPC_ENV_PLANES) ? e->planes : nullptr, nullptr, k_all,
                     (which & FPC_ENV_MASK) ? e->mask : nullptr, 0, e->stream);
}

int fpc_env_playout_step(fpc_env *e, uint64_t seed, const uint8_t *h_start, int max_plies, uint64_t game_stride, int which,
                         int k_all) {
  DevGuard guard_;
  int rc = env_check(e, "fpc_env_playout_step", guard_);
  if (rc != FPC_OK) return rc;
  if (!h_start) return fail(FPC_ERR_ARG, "fpc_env_playout_step: null start record");
  CK(cudaMemcpyAsync(e->start, h_start, e->rec, cudaMemcpyHostToDevice, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return fpc_playout_step(e->R, e->boards, e->n, seed, e->game, e->ply, e->start, max_plies, game_stride, nullptr, e->counts,
                          e->status, (which & FPC_ENV_PLANES) ? e->planes : nullptr, nullptr, k_all,
                          (which & FPC_ENV_MASK) ? e->mask : nullptr, e->counters, 0, e->stream);
}

struct EnvExport {
  DLManagedTensor t;
  int64_t shape[4];
  fpc_env *env;
};
static void env_export_deleter(DLManagedTensor *self) {
  if (!self) return;
  EnvExport *x = static_cast<EnvExport *>(self->manager_ctx);
  fpc_env *e = x->env;
  delete x;
  env_release(e);
}

DLManagedTensor *fpc_env_dlpack(fpc_env *e, int which) {
  DevGuard guard_;
  if (env_check(e, "fpc_env_dlpack", guard_) != FPC_OK) return nullptr;
  EnvExport *x = new EnvExport();
  memset(x, 0, sizeof *x);
  DLTensor &d = x->t.dl_tensor;
  const int R = e->R, A = fpc_num_action_channels(R);
  d.shape = x->shape;
  d.shape[0] = e->n;
  d.ndim = 1;
  switch (which) {
    case FPC_ENV_BOARDS: d.data = e->boards, d.dtype = {kDLUInt, 8, 1}, d.ndim = 2, d.shape[1] = e->rec; break;
    case FPC_ENV_COUNTS: d.data = e->counts, d.dtype = {kDLInt, 32, 1}; break;
    case FPC_ENV_STATUS: d.data = e->status, d.dtype = {kDLInt, 32, 1}; break;
    case FPC_ENV_PLY: d.data = e->ply, d.dtype = {kDLInt, 32, 1}; break;
    case FPC_ENV_GAME: d.data = e->game, d.dtype = {kDLInt, 64, 1}; break;
    case FPC_ENV_MOVES: d.data = e->moves, d.dtype = {kDLInt, 64, 1}, d.ndim = 2, d.shape[1] = FPC_MAX_MOVES; break;
    case FPC_ENV_FLAT: d.data = e->flat, d.dtype = {kDLInt, 32, 1}, d.ndim = 2, d.shape[1] = FPC_MAX_MOVES; break;
    case FPC_ENV_PLANES:
      d.data = e->planes, d.dtype = {kDLFloat, 32, 1}, d.ndim = 4, d.shape[1] = FPC_NUM_STATE_CHANNELS, d.shape[2] = d.shape[3] = R;
      break;
    case FPC_ENV_MASK: d.data = e->mask, d.dtype = {kDLFloat, 32, 1}, d.ndim = 4, d.shape[1] = A, d.shape[2] = d.shape[3] = R; break;
    default:
      delete x;
      fail(FPC_ERR_ARG, "fpc_env_dlpack: `which` must be exactly one FPC_ENV_* tensor");
      return nullptr;
  }
  d.device = {kDLCUDA, e->device};
  d.strides = nullptr;
  d.byte_offset = 0;
  x->env = e;
  x->t.manager_ctx = x;
  x->t.deleter = env_export_deleter;
  __atomic_add_fetch(&e->refs, 1, __ATOMIC_ACQ_REL);
  return &x->t;
}

}  // extern "C"
