// Batched PUCT (select / expand / backup) for sm_100a: one warp owns one game's tree in HBM.
// Boundary and array layout: include/fpc.h (struct fpc_tree).  Semantics follow the reference's
// fpchess::Node (src/cpp/node.{h,cpp}) driven by src/py/mcts.py; each routine cites the lines.
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include <cfloat>
#include <cmath>
#include <string>
#include <type_traits>

#include "../../include/fpc.h"
#include "fpc_device.cuh"
#include "fpc_host.h"

namespace fpc {

constexpr int SEL_WARPS = 4;
constexpr int ERR_NODE_CAP = 1, ERR_BOARD_CAP = 2, ERR_NO_CHILD = 4, ERR_MOVE = 8;

// A fresh root for game g: node 0 = `root` (one record), visit_count 1, no children; per-game state cleared.  Run by
// every thread of one CTA.
template <class G>
__device__ __forceinline__ void write_fresh_root(const fpc_tree &T, int g, const uint8_t *root) {
  const size_t slab = (size_t)g * T.node_cap;
  if (threadIdx.x == 0) {
    T.parent[slab] = -1;
    T.first_child[slab] = 0;
    T.n_children[slab] = 0;
    T.visits[slab] = 1;  // mcts.py:30
    T.move_flat[slab] = -1;
    T.board_idx[slab] = 0;
    T.value_sum[slab] = 0.0;
    T.prior[slab] = 0.0f;
    T.n_nodes[g] = 1;
    T.n_boards[g] = 1;
    T.leaf[g] = -1;
    T.dropped[g] = 0;
    T.error[g] = 0;
  }
  for (int i = threadIdx.x; i < G::REC; i += blockDim.x) T.boards[(size_t)g * T.board_cap * G::REC + i] = root[i];
}

template <class G>
__global__ void __launch_bounds__(256) tree_reset_kernel(const fpc_tree T, const uint8_t *roots) {
  write_fresh_root<G>(T, blockIdx.x, roots + (size_t)blockIdx.x * G::REC);
}

// ---- re-rooting on the played move (fpc_tree_advance), one CTA per game -------------------------------------------
// Invariants of a slab written by the kernels of this file, which the in-place compaction relies on:
//  (1) parent[i] < i for every node but the root: children are appended at n_nodes when their parent is expanded;
//  (2) hence the new root c has the smallest index of its subtree, and renumbering the kept nodes in ascending order of
//      their old index maps c to 0 and never raises an index (new <= old);
//  (3) a node is materialised before it can be expanded, so c's board slot, when it has one, is the smallest among the
//      subtree's boards and lands in slot 0; a c without a board was never selected and has no descendants.
// A gather in ascending chunks of old indices, each chunk read completely before a barrier and written after it, is
// therefore safe in place: every write lands at or below the chunk it came from, never on an entry not yet read.
// The old -> new map is a bitmap of the kept entries plus an exclusive prefix count per 32-entry word in dynamic shared
// memory (node_cap / 4 bytes); after the nodes it is rebuilt over the board slots.
constexpr int ADV_THREADS = 256, ADV_WARPS = ADV_THREADS / 32;
constexpr int ADV_ITEMS = 4;                          // nodes per thread and chunk: four independent loads in flight
constexpr int ADV_CHUNK = ADV_THREADS * ADV_ITEMS;    // 1,024 nodes = 32 map words

__device__ __forceinline__ bool map_bit(const uint32_t *bits, int b) { return (bits[b >> 5] >> (b & 31)) & 1u; }

// new index of kept entry b = the number of kept entries below it
__device__ __forceinline__ int map_rank(const uint32_t *bits, const uint32_t *pre, int b) {
  return (int)pre[b >> 5] + __popc(bits[b >> 5] & ((1u << (b & 31)) - 1u));
}

// pre[w] = exclusive prefix sum of popc(bits[w]) for w < nw; returns the total to every thread
__device__ int scan_map(const uint32_t *bits, uint32_t *pre, int nw, int *red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int carry = 0;
  for (int base = 0; base < nw; base += ADV_THREADS) {
    const int w = base + threadIdx.x;
    const int v = w < nw ? __popc(bits[w]) : 0;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(FULL, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) red[warp] = x;
    __syncthreads();
    int before = 0, tot = 0;
#pragma unroll
    for (int k = 0; k < ADV_WARPS; ++k) {
      const int n = red[k];
      before += k < warp ? n : 0;
      tot += n;
    }
    if (w < nw) pre[w] = carry + before + x - v;
    carry += tot;
    __syncthreads();
  }
  return carry;
}

template <class G>
__global__ void __launch_bounds__(ADV_THREADS) tree_advance_kernel(const fpc_tree T, const int32_t *actions, const uint8_t *roots,
                                                                   int max_nodes, int max_boards, int32_t *kept_out) {
  extern __shared__ uint32_t s_map[];  // [map_words] bits, then [map_words] prefix counts
  __shared__ int red[ADV_WARPS];
  __shared__ int s_c, s_mat;
  const int map_words = (T.node_cap + 31) >> 5;
  uint32_t *bits = s_map, *pre = s_map + map_words;
  const int g = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t slab = (size_t)g * T.node_cap;
  const uint8_t *root = roots + (size_t)g * G::REC;
  uint4 *pool = reinterpret_cast<uint4 *>(T.boards + (size_t)g * T.board_cap * G::REC);
  constexpr int V = G::REC / 16;  // 16-byte words per record
  const int action = actions[g];
  const int nn = T.n_nodes[g], nb_old = T.n_boards[g];
  const int nc0 = T.n_children[slab], fc0 = T.first_child[slab];
  if (tid == 0) s_c = -1, s_mat = 0;
  __syncthreads();
  // 1. c = the root child that made the move (the flat indices of siblings are unique: promotions share one child)
  if (action >= 0)
    for (int i = tid; i < nc0; i += ADV_THREADS)
      if (T.move_flat[slab + fc0 + i] == action) s_c = fc0 + i;
  __syncthreads();
  const int c = s_c;
  bool keep = c > 0;
  int c_slot = -1;
  if (keep) {  // uniform over the CTA
    // c's board, when it has one, must be the caller's position (a full move with promotion is not the index-built one)
    c_slot = T.board_idx[slab + c];
    bool diff = false;
    if (c_slot >= 0)
      for (int i = tid; i < V; i += ADV_THREADS) {
        const uint4 a = pool[(size_t)c_slot * V + i], b = reinterpret_cast<const uint4 *>(root)[i];
        diff |= a.x != b.x || a.y != b.y || a.z != b.z || a.w != b.w;
      }
    keep = !__syncthreads_or(diff);
  }
  // 2. subtree membership over [c, nn) (offsets r = i - c), in ascending chunks: a node's parent lies in an earlier chunk
  //    (its bit is final) or in this one, where the walk climbs on until it leaves the chunk or meets c.  Every warp's
  //    ballot is one map word.
  const int span = keep ? nn - c : 0;
  for (int base = 0; base < span; base += ADV_CHUNK) {
    int par[ADV_ITEMS], bix[ADV_ITEMS];
#pragma unroll
    for (int q = 0; q < ADV_ITEMS; ++q) {
      const int r = base + q * ADV_THREADS + tid;
      par[q] = r < span ? T.parent[slab + c + r] : -1;
      bix[q] = r < span ? T.board_idx[slab + c + r] : -1;
    }
    int n_mat = 0;
#pragma unroll
    for (int q = 0; q < ADV_ITEMS; ++q) {
      const int r = base + q * ADV_THREADS + tid;
      bool in = r == 0;
      if (r > 0 && r < span) {
        int p = par[q];
        while (p >= c + base && p != c) p = T.parent[slab + p];
        in = p == c || (p > c && map_bit(bits, p - c));
      }
      const unsigned w = __ballot_sync(FULL, in);
      n_mat += __popc(__ballot_sync(FULL, in && bix[q] >= 0));
      const int word = (base + q * ADV_THREADS) / 32 + warp;
      if (lane == 0 && word * 32 < span) bits[word] = w;
    }
    if (lane == 0 && n_mat) atomicAdd(&s_mat, n_mat);
    __syncthreads();
  }
  int kept = 0;
  if (keep) {
    kept = scan_map(bits, pre, (span + 31) >> 5, red);
    keep = kept <= max_nodes && s_mat <= max_boards;
  }
  if (!keep) {  // every read of the old tree is behind a barrier by now
    write_fresh_root<G>(T, g, root);
    if (tid == 0 && kept_out) kept_out[g] = 0;
    return;
  }
  // 3. gather the kept nodes in place; parent and first_child through the map, the rest unchanged but for the root
  for (int base = 0; base < span; base += ADV_CHUNK) {
    int dst[ADV_ITEMS], par[ADV_ITEMS], fc[ADV_ITEMS], nch[ADV_ITEMS], vis[ADV_ITEMS], mv[ADV_ITEMS], bix[ADV_ITEMS];
    double vs[ADV_ITEMS];
    float pr[ADV_ITEMS];
#pragma unroll
    for (int q = 0; q < ADV_ITEMS; ++q) {
      const int r = base + q * ADV_THREADS + tid;
      dst[q] = -1;
      if (r < span && map_bit(bits, r)) {
        const size_t i = slab + c + r;
        dst[q] = map_rank(bits, pre, r);
        par[q] = T.parent[i], fc[q] = T.first_child[i], nch[q] = T.n_children[i], vis[q] = T.visits[i];
        mv[q] = T.move_flat[i], bix[q] = T.board_idx[i], vs[q] = T.value_sum[i], pr[q] = T.prior[i];
      }
    }
#pragma unroll
    for (int q = 0; q < ADV_ITEMS; ++q) {
      if (dst[q] < 0) continue;
      if (dst[q] == 0) {
        par[q] = -1, mv[q] = -1, pr[q] = 0.0f;
      } else {
        par[q] = map_rank(bits, pre, par[q] - c);
      }
      fc[q] = nch[q] > 0 ? map_rank(bits, pre, fc[q] - c) : 0;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < ADV_ITEMS; ++q) {
      if (dst[q] < 0) continue;
      const size_t j = slab + dst[q];
      T.parent[j] = par[q], T.first_child[j] = fc[q], T.n_children[j] = nch[q], T.visits[j] = vis[q];
      T.move_flat[j] = mv[q], T.board_idx[j] = bix[q], T.value_sum[j] = vs[q], T.prior[j] = pr[q];
    }
    __syncthreads();
  }
  // 4. boards: the map is rebuilt over the slots the kept nodes own and the boards gathered the same way.  An
  //    unmaterialised c owns none of them; it gets the caller's board in slot 0 and every kept slot moves up by one.
  const int off = c_slot < 0;
  const int n_slots = min(nb_old, map_words * 32);
  const int slot_words = (n_slots + 31) >> 5;
  for (int w = tid; w < slot_words; w += ADV_THREADS) bits[w] = 0;
  __syncthreads();
  for (int j = tid; j < kept; j += ADV_THREADS) {
    const int b = T.board_idx[slab + j];
    if (b >= 0 && b < n_slots) atomicOr(&bits[b >> 5], 1u << (b & 31));
  }
  __syncthreads();
  const int kept_boards = scan_map(bits, pre, slot_words, red);
  for (int j = tid; j < kept; j += ADV_THREADS) {
    const int b = T.board_idx[slab + j];
    T.board_idx[slab + j] = j == 0 ? 0 : b >= 0 ? off + map_rank(bits, pre, b) : -1;
  }
  constexpr int BPC = ADV_THREADS / V;  // boards per chunk
  for (int base = 0; base < n_slots; base += BPC) {
    const int s = base + tid / V, part = tid % V;
    int dst = -1;
    uint4 v;
    if (tid < BPC * V && s < n_slots && map_bit(bits, s)) {
      v = pool[(size_t)s * V + part];
      dst = off + map_rank(bits, pre, s);
    }
    __syncthreads();
    if (dst >= 0) pool[(size_t)dst * V + part] = v;
    __syncthreads();
  }
  if (off)
    for (int i = tid; i < V; i += ADV_THREADS) pool[i] = reinterpret_cast<const uint4 *>(root)[i];
  if (tid == 0) {
    T.n_nodes[g] = kept;
    T.n_boards[g] = kept_boards + off;
    T.leaf[g] = -1;
    T.dropped[g] = 0;
    T.error[g] = 0;
    if (kept_out) kept_out[g] = kept;
  }
}

// descend's default step below the root: Node::SelectChild.
struct SelectChild {};

// Node::ChooseLeaf's descent (node.cpp:21-26) + Node::SelectChild (node.cpp:49-78), then the leaf's board materialised
// into leaf_boards.  One warp of game g; `b` is the warp's 256-byte record scratch in shared memory.  root_step(node, nc,
// fc, nv) may replace the root's step: it receives the root (node 0) and its (n_children, first_child, visits), may move
// them to the node the descent continues from, and returns false when it has dropped the game.  step(node, nc, fc, nv)
// may replace every later step in the same way, at a node with nc > 0 children; the default is SelectChild, spelled out
// in the loop below.
template <class G, class RootStep, class Step = SelectChild>
__device__ __forceinline__ void descend(const fpc_tree &T, int g, int lane, uint8_t *b, RootStep root_step, Step step = {}) {
  const size_t slab = (size_t)g * T.node_cap;
  const int32_t *visits = T.visits + slab, *first_child = T.first_child + slab, *n_children = T.n_children + slab;
  const double *value_sum = T.value_sum + slab;
  const float *prior = T.prior + slab;
  // One dependent memory round per level: while scanning the children of `node` every lane also fetches
  // its child's own child range, and the winner's (first_child, n_children, visits) travel with the arg-max.
  int node = 0;
  int nc = n_children[0], fc = first_child[0], nv = visits[0];
  if (!root_step(node, nc, fc, nv)) return;
  while (nc > 0) {
    if constexpr (!std::is_same_v<Step, SelectChild>) {
      if (!step(node, nc, fc, nv)) return;
      continue;
    }
    const double lg = log(sqrt((double)nv));
    double best = -CUDART_INF;
    int best_i = 0x7fffffff, b_nc = 0, b_fc = 0, b_nv = 0;
    for (int i = lane; i < nc; i += 32) {
      const int n = visits[fc + i];
      const int c_nc = n_children[fc + i], c_fc = first_child[fc + i];
      const double q = n > 0 ? value_sum[fc + i] / (double)n : 0.0;
      const double ucb = q + T.C * sqrt(lg / (double)(1 + n)) * (double)prior[fc + i];
      if (ucb > best) {  // strict: the first maximum wins
        best = ucb;
        best_i = i;
        b_nc = c_nc, b_fc = c_fc, b_nv = n;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ob = __shfl_xor_sync(FULL, best, o);
      const int oi = __shfl_xor_sync(FULL, best_i, o);
      const int o_nc = __shfl_xor_sync(FULL, b_nc, o), o_fc = __shfl_xor_sync(FULL, b_fc, o), o_nv = __shfl_xor_sync(FULL, b_nv, o);
      if (oi != 0x7fffffff && (best_i == 0x7fffffff || ob > best || (ob == best && oi < best_i))) {
        best = ob;
        best_i = oi;
        b_nc = o_nc, b_fc = o_fc, b_nv = o_nv;
      }
    }
    if (best_i == 0x7fffffff) {  // "Failed to select a child." (node.cpp:72-75)
      if (lane == 0) {
        T.error[g] |= ERR_NO_CHILD;
        T.leaf[g] = -1;
        T.dropped[g] = 1;
      }
      return;
    }
    node = fc + best_i;
    nc = b_nc, fc = b_fc, nv = b_nv;
  }
  // materialise the leaf's board: parent's board + MakeMove(Move(flat_index)) (node.cpp:87-92)
  uint8_t *pool = T.boards + (size_t)g * T.board_cap * G::REC;
  int bi = T.board_idx[slab + node];
  if (bi < 0) {
    const int pb = T.board_idx[slab + T.parent[slab + node]];
    if (lane < G::REC / 16) reinterpret_cast<uint4 *>(b)[lane] = reinterpret_cast<const uint4 *>(pool + (size_t)pb * G::REC)[lane];
    __syncwarp();
    int ok = 1;
    if (lane == 0) {
      int from, to;
      decode_flat_move<G>(T.move_flat[slab + node], from, to);
      ok = apply_move_record<G>(b, from, to, NO_PIECE, G::NSQ, G::NSQ, 0) ? 1 : 0;
    }
    ok = __shfl_sync(FULL, ok, 0);
    bi = T.n_boards[g];
    if (bi >= T.board_cap || !ok) {
      if (lane == 0) {
        T.error[g] |= ok ? ERR_BOARD_CAP : ERR_MOVE;
        T.leaf[g] = -1;
        T.dropped[g] = 1;
      }
      return;
    }
    __syncwarp();
    if (lane < G::REC / 16) reinterpret_cast<uint4 *>(pool + (size_t)bi * G::REC)[lane] = reinterpret_cast<const uint4 *>(b)[lane];
    if (lane == 0) {
      T.board_idx[slab + node] = bi;
      T.n_boards[g] = bi + 1;
    }
  } else {
    if (lane < G::REC / 16) reinterpret_cast<uint4 *>(b)[lane] = reinterpret_cast<const uint4 *>(pool + (size_t)bi * G::REC)[lane];
    __syncwarp();
  }
  if (lane < G::REC / 16) reinterpret_cast<uint4 *>(T.leaf_boards + (size_t)g * G::REC)[lane] = reinterpret_cast<const uint4 *>(b)[lane];
  if (lane == 0) {
    T.leaf[g] = node;
    T.k[g] = b[G::OFF_TURN] & 3;
  }
}

template <class G>
__global__ void __launch_bounds__(SEL_WARPS * 32) tree_descend_kernel(const fpc_tree T) {
  __shared__ alignas(16) uint8_t recs[SEL_WARPS][256];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * SEL_WARPS + wib;
  if (g >= T.n_games) return;
  if (T.dropped[g]) {
    if (lane == 0) T.leaf[g] = -1;
    return;
  }
  descend<G>(T, g, lane, recs[wib], [](int &, int &, int &, int &) { return true; });
}

// The reference rotates a whole leaf batch by the colour of states[0] (src/cpp/board.cpp:354-355,
// mcts.py:69), states = the leaves that are NOT terminal (mcts.py:18-26 drops terminal leaves before the batch is
// built): k[g] <- side to move of the first leaf whose status (already computed) says IN_PROGRESS.
template <class G>
__global__ void __launch_bounds__(1024) tree_batch_k_kernel(const fpc_tree T) {
  __shared__ int first;
  if (threadIdx.x == 0) first = 0x7fffffff;
  __syncthreads();
  int mine = 0x7fffffff;
  for (int g = threadIdx.x; g < T.n_games; g += blockDim.x)
    if (T.leaf[g] >= 0 && (T.leaf_status[g] & FPC_STATUS_RESULT_MASK) == 0) {
      mine = g;
      break;
    }
  if (mine != 0x7fffffff) atomicMin(&first, mine);
  __syncthreads();
  if (first == 0x7fffffff) return;
  const int k = T.leaf_boards[(size_t)first * G::REC + G::OFF_TURN] & 3;
  for (int g = threadIdx.x; g < T.n_games; g += blockDim.x) T.k[g] = k;
}

// mcts.py:66-79 + 82-89 and node.cpp:33-43,133-154, one CTA per game.
constexpr int EXP_THREADS = 256;  // 8 CTAs per SM: 1,024 games are one wave on 148 SMs
constexpr int EXP_WARPS = EXP_THREADS / 32;

// online soft-max statistics: running maximum m and sum s of exp(x - m)
__device__ __forceinline__ void softmax_merge(float &m, float &s, float om, float os) {
  const float nm = fmaxf(m, om);
  s = (m == nm ? s : s * __expf(m - nm)) + (om == nm ? os : os * __expf(om - nm));
  m = nm;
}

template <class G>
__global__ void __launch_bounds__(EXP_THREADS, 8) tree_expand_backup_kernel(const fpc_tree T, const float *logits, const float *values) {
  __shared__ float red_m[EXP_WARPS], red_s[EXP_WARPS];
  __shared__ double red_d[EXP_WARPS];
  __shared__ int red_i[EXP_WARPS];
  __shared__ float s_max, s_sum;
  __shared__ double s_msum;
  __shared__ int s_base;
  constexpr int ANC_MAX = 64;
  __shared__ int s_anc[ANC_MAX];
  __shared__ int s_nanc, s_anc_next;
  const int g = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // every per-game scalar is requested at once (one memory latency instead of a chain of them), and so are the legal
  // moves (rows past the count hold stale moves of earlier leaves: valid memory, ignored below)
  const int leaf = T.leaf[g];
  const int status = T.leaf_status[g];
  const int cnt = T.leaf_counts[g];
  const int k = T.k[g] & 3;
  const float value_in = values[g];
  constexpr int PER = (MAX_MOVES + EXP_THREADS - 1) / EXP_THREADS;
  int flat_in[PER], prev_in[PER];
#pragma unroll
  for (int q = 0; q < PER; ++q) {
    const int i = tid + q * EXP_THREADS;
    flat_in[q] = i < MAX_MOVES ? T.leaf_flat[(size_t)g * MAX_MOVES + i] : -1;
    prev_in[q] = (i > 0 && i < MAX_MOVES) ? T.leaf_flat[(size_t)g * MAX_MOVES + i - 1] : -1;
  }
  if (leaf < 0) return;
  const size_t slab = (size_t)g * T.node_cap;
  // The latency-bound tail is prepared while the logits stream: one thread (of the last warp) walks the leaf's ancestors
  // now -- a chain of dependent loads -- so that the backup at the end is one parallel round of updates; thread 0 has
  // the node count of the slab in a register by then.
  if (tid == EXP_THREADS - 32) {
    int node = leaf, cnt = 0;
    while (node >= 0 && cnt < ANC_MAX) {
      s_anc[cnt++] = node;
      node = T.parent[slab + node];
    }
    s_nanc = cnt;
    s_anc_next = node;  // >= 0 only for a path longer than ANC_MAX
  }
  const int nodes_before = tid == 0 ? T.n_nodes[g] : 0;
  const int result = status & FPC_STATUS_RESULT_MASK;
  float value;
  if (result != 0) {
    // terminal leaf: Backpropagate(0) for a stalemate, Backpropagate(-1) for any win; the root drops out
    value = result == 3 ? 0.0f : -1.0f;
    if (tid == 0) T.dropped[g] = 1;
  } else {
    value = value_in;
    const float *lg = logits + (size_t)g * G::ASZ;
    // ---- the legal moves' own logits are requested first (scattered, ~20 of them) ---------------------
    int flat[PER];
    float lgt[PER];
    bool first[PER];
#pragma unroll
    for (int q = 0; q < PER; ++q) {
      const int i = tid + q * EXP_THREADS;
      flat[q] = -1, lgt[q] = 0.0f, first[q] = false;
      if (i < cnt) {
        flat[q] = flat_in[q];
        first[q] = i == 0 || prev_in[q] != flat[q];  // promotions share an index
        if (first[q]) {
          // policy[plane][r][c] = rot90(net_out, -k)[plane][r][c]: one clockwise quarter turn reads out[i][j] = in[R-1-j][i]
          const int plane = flat[q] / G::NSQ, sq = flat[q] - plane * G::NSQ;
          int r = sq / G::R, c = sq - r * G::R;
          for (int t = 0; t < k; ++t) {
            const int nr = G::R - 1 - c;
            c = r;
            r = nr;
          }
          lgt[q] = __ldg(lg + plane * G::NSQ + r * G::R + c);
        }
      }
    }
    // ---- softmax over the whole action space (mcts.py:67): ONE streaming pass, online max / sum; four independent
    //      16-byte loads per thread and iteration keep enough bytes in flight to stream at the HBM rate.  The running
    //      maximum starts at -FLT_MAX, not -inf: a group of -inf logits (a masked policy) then rescales by
    //      exp(-inf - -FLT_MAX) = 0 instead of exp(-inf - -inf) = NaN, and -inf entries get a zero prior ----------
    float m = -FLT_MAX, s = 0.0f;
    const float4 *lg4 = reinterpret_cast<const float4 *>(lg);
    constexpr int N4 = G::ASZ / 4;
    int i = tid;
    for (; i + 3 * EXP_THREADS < N4; i += 4 * EXP_THREADS) {
      const float4 a = __ldcs(lg4 + i), b = __ldcs(lg4 + i + EXP_THREADS), c = __ldcs(lg4 + i + 2 * EXP_THREADS),
                   d = __ldcs(lg4 + i + 3 * EXP_THREADS);
      const float mx = fmaxf(fmaxf(fmaxf(fmaxf(a.x, a.y), fmaxf(a.z, a.w)), fmaxf(fmaxf(b.x, b.y), fmaxf(b.z, b.w))),
                             fmaxf(fmaxf(fmaxf(c.x, c.y), fmaxf(c.z, c.w)), fmaxf(fmaxf(d.x, d.y), fmaxf(d.z, d.w))));
      const float nm = fmaxf(m, mx);
      s = s * __expf(m - nm) + ((__expf(a.x - nm) + __expf(a.y - nm)) + (__expf(a.z - nm) + __expf(a.w - nm))) +
          ((__expf(b.x - nm) + __expf(b.y - nm)) + (__expf(b.z - nm) + __expf(b.w - nm))) +
          ((__expf(c.x - nm) + __expf(c.y - nm)) + (__expf(c.z - nm) + __expf(c.w - nm))) +
          ((__expf(d.x - nm) + __expf(d.y - nm)) + (__expf(d.z - nm) + __expf(d.w - nm)));
      m = nm;
    }
    for (; i < N4; i += EXP_THREADS) {
      const float4 a = __ldcs(lg4 + i);
      const float nm = fmaxf(m, fmaxf(fmaxf(a.x, a.y), fmaxf(a.z, a.w)));
      s = s * __expf(m - nm) + ((__expf(a.x - nm) + __expf(a.y - nm)) + (__expf(a.z - nm) + __expf(a.w - nm)));
      m = nm;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) softmax_merge(m, s, __shfl_xor_sync(FULL, m, o), __shfl_xor_sync(FULL, s, o));
    if (lane == 0) {
      red_m[warp] = m;
      red_s[warp] = s;
    }
    __syncthreads();
    if (tid == 0) {
      float M = red_m[0];
      for (int w = 1; w < EXP_WARPS; ++w) M = fmaxf(M, red_m[w]);
      double S = 0.0;
      for (int w = 0; w < EXP_WARPS; ++w)
        if (red_s[w] > 0.0f) S += (double)red_s[w] * (double)expf(red_m[w] - M);
      s_max = M;
      s_sum = (float)S;
    }
    __syncthreads();
    // ---- legal moves: un-rotated above; mask, renormalise (mcts.py:69-76) ---------------------------------
    float p[PER];
    double psum = 0.0;
#pragma unroll
    for (int q = 0; q < PER; ++q) {
      p[q] = first[q] ? expf(lgt[q] - s_max) / s_sum : 0.0f;
      psum += (double)p[q];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) psum += __shfl_xor_sync(FULL, psum, o);
    if (lane == 0) red_d[warp] = psum;
    __syncthreads();
    if (tid == 0) {
      double t = 0.0;
      for (int w = 0; w < EXP_WARPS; ++w) t += red_d[w];
      s_msum = t;
    }
    __syncthreads();
    // ---- one child per non-zero prior, ascending flat index (mcts.py:83-87, node.cpp:79-98): move i = tid + q*THREADS,
    //      so the children of slice q come after every child of slice q-1 -------------------------------------------
    int base_q = 0;
    bool capped = false;
#pragma unroll
    for (int q = 0; q < PER; ++q) {
      const float prior = (float)((double)p[q] / s_msum);
      const bool make = first[q] && prior != 0.0f;
      const unsigned bal = __ballot_sync(FULL, make);
      if (lane == 0) red_i[warp] = __popc(bal);
      __syncthreads();
      int before = 0, tot = 0;
      for (int w = 0; w < EXP_WARPS; ++w) {
        const int c = red_i[w];
        if (w < warp) before += c;
        tot += c;
      }
      if (q == 0) {
        // the total number of children is needed up front: count the later slices too
        int all = tot;
#pragma unroll
        for (int q2 = 1; q2 < PER; ++q2) {
          const float pr2 = (float)((double)p[q2] / s_msum);
          all += __syncthreads_count(first[q2] && pr2 != 0.0f);
        }
        if (tid == 0) {
          int base = nodes_before;
          if (base + all > T.node_cap) {
            T.error[g] |= ERR_NODE_CAP;
            base = -1;
          } else {
            T.n_nodes[g] = base + all;
            T.first_child[slab + leaf] = base;
            T.n_children[slab + leaf] = all;
          }
          s_base = base;
        }
        __syncthreads();
        capped = s_base < 0;
      }
      if (make && !capped) {
        const size_t c = slab + s_base + base_q + before + __popc(bal & ((1u << lane) - 1u));
        T.parent[c] = leaf;
        T.first_child[c] = 0;
        T.n_children[c] = 0;
        T.visits[c] = 1;  // node.h:28
        T.move_flat[c] = flat[q];
        T.board_idx[c] = -1;
        T.value_sum[c] = 0.0;
        T.prior[c] = prior;
      }
      base_q += tot;
      __syncthreads();
    }
  }
  // ---- Node::Backpropagate (node.cpp:133-142): +v at the leaf, sign flips at every ancestor ------
  __syncthreads();  // the ancestor list is complete (and, when expanding, every child has been written)
  if (tid < s_nanc) {
    const int node = s_anc[tid];
    T.value_sum[slab + node] += (tid & 1) ? -(double)value : (double)value;
    T.visits[slab + node] += 1;
  }
  if (tid == 0 && s_anc_next >= 0) {  // deeper than ANC_MAX: the rest of the path one by one
    double v = (ANC_MAX & 1) ? -(double)value : (double)value;
    int node = s_anc_next;
    while (node >= 0) {
      T.value_sum[slab + node] += v;
      T.visits[slab + node] += 1;
      v = -v;
      node = T.parent[slab + node];
    }
  }
}

// ---- leaf-parallel PUCT (fpc_tree_select_leaves / fpc_tree_expand_backup_leaves; semantics in include/fpc.h) -------
constexpr int LB_PATH = 64;  // path nodes a descent keeps in shared memory for its marks; deeper ones are re-walked

// The L slots of game g, one after the other: slot j must see the marks of slots < j.  Each level is one memory round
// as in tree_descend_kernel, with in_flight read beside visits; after the first descent the upper levels come from the
// cache.  root_step(node, depth, nc, fc, nv) may replace the root's step: it receives the root (node 0, depth 0) with its
// effective (n_children, first_child, visits), may move them to a child (recording it in path[depth]) and returns 0 or
// the error bits that end the game.  step(node, nc, fc) may replace SelectChild at every later node with nc > 0
// children: it returns the chosen child's index or -1.  Returns the number of slots that were filled.
template <class G, class RootStep, class Step = SelectChild>
__device__ __forceinline__ int leaves_select(const fpc_tree &T, const fpc_leaf_batch &B, int g, int lane, uint8_t *b, int *path,
                                             RootStep root_step, Step step = {}) {
  const int L = B.L, VL = B.virtual_loss;
  const size_t s0 = (size_t)g * L, slab = (size_t)g * T.node_cap;
  const int32_t *visits = T.visits + slab, *first_child = T.first_child + slab, *n_children = T.n_children + slab;
  const double *value_sum = T.value_sum + slab;
  const float *prior = T.prior + slab;
  int32_t *in_flight = B.in_flight + slab;
  uint8_t *pool = T.boards + (size_t)g * T.board_cap * G::REC;
  int n_boards = T.n_boards[g], n_coll = 0, j = 0;
  bool live = !T.dropped[g];
  if (lane == 0) T.leaf[g] = -1;
  for (; live && j < L; ++j) {
    int node = 0, depth = 0;
    int nc = n_children[0], fc = first_child[0], nv = visits[0] + VL * in_flight[0];
    if (lane == 0) path[0] = 0;
    int err = root_step(node, depth, nc, fc, nv);
    while (!err && nc > 0) {
      if constexpr (!std::is_same_v<Step, SelectChild>) {
        const int i = step(node, nc, fc);
        if (i < 0) {
          err = ERR_NO_CHILD;
          break;
        }
        node = fc + i;
        ++depth;
        if (lane == 0 && depth < LB_PATH) path[depth] = node;
        nc = n_children[node], fc = first_child[node];
        continue;
      }
      const double lg = log(sqrt((double)nv));
      double best = -CUDART_INF;
      int best_i = 0x7fffffff, b_nc = 0, b_fc = 0, b_nv = 0;
      for (int i = lane; i < nc; i += 32) {
        const int vl = VL * in_flight[fc + i];
        const int n = visits[fc + i] + vl;
        const int c_nc = n_children[fc + i], c_fc = first_child[fc + i];
        const double q = n > 0 ? (value_sum[fc + i] - (double)vl) / (double)n : 0.0;
        const double ucb = q + T.C * sqrt(lg / (double)(1 + n)) * (double)prior[fc + i];
        if (ucb > best) {  // strict: the first maximum wins
          best = ucb;
          best_i = i;
          b_nc = c_nc, b_fc = c_fc, b_nv = n;
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double ob = __shfl_xor_sync(FULL, best, o);
        const int oi = __shfl_xor_sync(FULL, best_i, o);
        const int o_nc = __shfl_xor_sync(FULL, b_nc, o), o_fc = __shfl_xor_sync(FULL, b_fc, o), o_nv = __shfl_xor_sync(FULL, b_nv, o);
        if (oi != 0x7fffffff && (best_i == 0x7fffffff || ob > best || (ob == best && oi < best_i))) {
          best = ob;
          best_i = oi;
          b_nc = o_nc, b_fc = o_fc, b_nv = o_nv;
        }
      }
      if (best_i == 0x7fffffff) {  // "Failed to select a child." (node.cpp:72-75)
        err = ERR_NO_CHILD;
        break;
      }
      node = fc + best_i;
      ++depth;
      if (lane == 0 && depth < LB_PATH) path[depth] = node;
      nc = b_nc, fc = b_fc, nv = b_nv;
    }
    const bool coll = !err && in_flight[node] > 0;
    if (!err) {
      int bi = T.board_idx[slab + node];
      if (bi < 0) {  // a LEAF reached for the first time (a collision's endpoint was materialised by an earlier slot)
        const int pb = T.board_idx[slab + T.parent[slab + node]];
        if (lane < G::REC / 16) reinterpret_cast<uint4 *>(b)[lane] = reinterpret_cast<const uint4 *>(pool + (size_t)pb * G::REC)[lane];
        __syncwarp();
        int ok = 1;
        if (lane == 0) {
          int from, to;
          decode_flat_move<G>(T.move_flat[slab + node], from, to);
          ok = apply_move_record<G>(b, from, to, NO_PIECE, G::NSQ, G::NSQ, 0) ? 1 : 0;
        }
        ok = __shfl_sync(FULL, ok, 0);
        bi = n_boards;
        if (bi >= T.board_cap || !ok) {
          err = ok ? ERR_BOARD_CAP : ERR_MOVE;
        } else {
          __syncwarp();
          if (lane < G::REC / 16) reinterpret_cast<uint4 *>(pool + (size_t)bi * G::REC)[lane] = reinterpret_cast<const uint4 *>(b)[lane];
          if (lane == 0) T.board_idx[slab + node] = bi;
          n_boards = bi + 1;
        }
      } else {
        if (lane < G::REC / 16) reinterpret_cast<uint4 *>(b)[lane] = reinterpret_cast<const uint4 *>(pool + (size_t)bi * G::REC)[lane];
        __syncwarp();
      }
    }
    if (err) {  // this slot and the later ones stay EMPTY; the earlier slots keep their marks
      if (lane == 0) {
        T.error[g] |= err;
        T.dropped[g] = 1;
      }
      live = false;
      break;
    }
    const size_t s = s0 + j;
    if (lane < G::REC / 16) reinterpret_cast<uint4 *>(B.leaf_boards + s * G::REC)[lane] = reinterpret_cast<const uint4 *>(b)[lane];
    if (lane == 0) {
      B.slot_node[s] = node;
      B.slot_kind[s] = coll ? FPC_SLOT_COLLISION : FPC_SLOT_LEAF;
      B.k[s] = b[G::OFF_TURN] & 3;
      if (j == 0 && !coll) T.leaf[g] = node;
    }
    n_coll += coll;
    // the marks: the first LB_PATH levels from shared memory in one round, a deeper rest by a walk up from the endpoint
    __syncwarp();
    const int top = min(depth, LB_PATH - 1);
    for (int i = lane; i <= top; i += 32) in_flight[path[i]] += 1;
    if (lane == 0 && depth > top)
      for (int x = node; x != path[top]; x = T.parent[slab + x]) in_flight[x] += 1;
    __syncwarp();  // the next descent reads these marks
  }
  for (int jj = j + lane; jj < L; jj += 32) {
    B.slot_node[s0 + jj] = -1;
    B.slot_kind[s0 + jj] = FPC_SLOT_EMPTY;
    B.k[s0 + jj] = 0;
  }
  if (lane == 0) {
    T.n_boards[g] = n_boards;
    if (n_coll) B.collisions[g] += n_coll;
  }
  return j;
}

template <class G>
__global__ void __launch_bounds__(SEL_WARPS * 32) leaves_descend_kernel(const fpc_tree T, const fpc_leaf_batch B) {
  __shared__ alignas(16) uint8_t recs[SEL_WARPS][256];
  __shared__ int paths[SEL_WARPS][LB_PATH];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * SEL_WARPS + wib;
  if (g >= T.n_games) return;
  leaves_select<G>(T, B, g, lane, recs[wib], paths[wib], [](int &, int &, int &, int &, int &) { return 0; });
}

// tree_batch_k_kernel over the slots: k <- side to move of the first LEAF slot whose status says IN_PROGRESS
template <class G>
__global__ void __launch_bounds__(1024) leaves_batch_k_kernel(const fpc_leaf_batch B, int n_slots) {
  __shared__ int first;
  if (threadIdx.x == 0) first = 0x7fffffff;
  __syncthreads();
  int mine = 0x7fffffff;
  for (int s = threadIdx.x; s < n_slots; s += blockDim.x)
    if (B.slot_kind[s] == FPC_SLOT_LEAF && (B.leaf_status[s] & FPC_STATUS_RESULT_MASK) == 0) {
      mine = s;
      break;
    }
  if (mine != 0x7fffffff) atomicMin(&first, mine);
  __syncthreads();
  if (first == 0x7fffffff) return;
  const int k = B.leaf_boards[(size_t)first * G::REC + G::OFF_TURN] & 3;
  for (int s = threadIdx.x; s < n_slots; s += blockDim.x) B.k[s] = k;
}

// Per-slot priors, one CTA per LEAF slot that is in progress: tree_expand_backup_kernel's soft-max, un-rotation, mask
// and renormalisation, statement for statement (so the priors are its bits), into B.priors[slot][i] for the legal
// entries i < count; 0 where no child is made (a repeated promotion index).
template <class G>
__global__ void __launch_bounds__(EXP_THREADS, 8) leaves_priors_kernel(const fpc_leaf_batch B, const float *logits) {
  __shared__ float red_m[EXP_WARPS], red_s[EXP_WARPS];
  __shared__ double red_d[EXP_WARPS];
  __shared__ float s_max, s_sum;
  __shared__ double s_msum;
  const size_t s = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (B.slot_kind[s] != FPC_SLOT_LEAF || (B.leaf_status[s] & FPC_STATUS_RESULT_MASK) != 0) return;
  const int cnt = B.leaf_counts[s];
  const int k = B.k[s] & 3;
  constexpr int PER = (MAX_MOVES + EXP_THREADS - 1) / EXP_THREADS;
  const float *lg = logits + s * G::ASZ;
  int flat[PER];
  float lgt[PER];
  bool first[PER];
#pragma unroll
  for (int q = 0; q < PER; ++q) {
    const int i = tid + q * EXP_THREADS;
    flat[q] = -1, lgt[q] = 0.0f, first[q] = false;
    if (i < cnt) {
      flat[q] = B.leaf_flat[s * MAX_MOVES + i];
      first[q] = i == 0 || B.leaf_flat[s * MAX_MOVES + i - 1] != flat[q];  // promotions share an index
      if (first[q]) {
        const int plane = flat[q] / G::NSQ, sq = flat[q] - plane * G::NSQ;
        int r = sq / G::R, c = sq - r * G::R;
        for (int t = 0; t < k; ++t) {
          const int nr = G::R - 1 - c;
          c = r;
          r = nr;
        }
        lgt[q] = __ldg(lg + plane * G::NSQ + r * G::R + c);
      }
    }
  }
  float m = -FLT_MAX, s_ = 0.0f;
  const float4 *lg4 = reinterpret_cast<const float4 *>(lg);
  constexpr int N4 = G::ASZ / 4;
  int i = tid;
  for (; i + 3 * EXP_THREADS < N4; i += 4 * EXP_THREADS) {
    const float4 a = __ldcs(lg4 + i), b = __ldcs(lg4 + i + EXP_THREADS), c = __ldcs(lg4 + i + 2 * EXP_THREADS),
                 d = __ldcs(lg4 + i + 3 * EXP_THREADS);
    const float mx = fmaxf(fmaxf(fmaxf(fmaxf(a.x, a.y), fmaxf(a.z, a.w)), fmaxf(fmaxf(b.x, b.y), fmaxf(b.z, b.w))),
                           fmaxf(fmaxf(fmaxf(c.x, c.y), fmaxf(c.z, c.w)), fmaxf(fmaxf(d.x, d.y), fmaxf(d.z, d.w))));
    const float nm = fmaxf(m, mx);
    s_ = s_ * __expf(m - nm) + ((__expf(a.x - nm) + __expf(a.y - nm)) + (__expf(a.z - nm) + __expf(a.w - nm))) +
         ((__expf(b.x - nm) + __expf(b.y - nm)) + (__expf(b.z - nm) + __expf(b.w - nm))) +
         ((__expf(c.x - nm) + __expf(c.y - nm)) + (__expf(c.z - nm) + __expf(c.w - nm))) +
         ((__expf(d.x - nm) + __expf(d.y - nm)) + (__expf(d.z - nm) + __expf(d.w - nm)));
    m = nm;
  }
  for (; i < N4; i += EXP_THREADS) {
    const float4 a = __ldcs(lg4 + i);
    const float nm = fmaxf(m, fmaxf(fmaxf(a.x, a.y), fmaxf(a.z, a.w)));
    s_ = s_ * __expf(m - nm) + ((__expf(a.x - nm) + __expf(a.y - nm)) + (__expf(a.z - nm) + __expf(a.w - nm)));
    m = nm;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) softmax_merge(m, s_, __shfl_xor_sync(FULL, m, o), __shfl_xor_sync(FULL, s_, o));
  if (lane == 0) {
    red_m[warp] = m;
    red_s[warp] = s_;
  }
  __syncthreads();
  if (tid == 0) {
    float M = red_m[0];
    for (int w = 1; w < EXP_WARPS; ++w) M = fmaxf(M, red_m[w]);
    double S = 0.0;
    for (int w = 0; w < EXP_WARPS; ++w)
      if (red_s[w] > 0.0f) S += (double)red_s[w] * (double)expf(red_m[w] - M);
    s_max = M;
    s_sum = (float)S;
  }
  __syncthreads();
  float p[PER];
  double psum = 0.0;
#pragma unroll
  for (int q = 0; q < PER; ++q) {
    p[q] = first[q] ? expf(lgt[q] - s_max) / s_sum : 0.0f;
    psum += (double)p[q];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) psum += __shfl_xor_sync(FULL, psum, o);
  if (lane == 0) red_d[warp] = psum;
  __syncthreads();
  if (tid == 0) {
    double t = 0.0;
    for (int w = 0; w < EXP_WARPS; ++w) t += red_d[w];
    s_msum = t;
  }
  __syncthreads();
#pragma unroll
  for (int q = 0; q < PER; ++q) {
    const int i = tid + q * EXP_THREADS;
    if (i < cnt) B.priors[s * MAX_MOVES + i] = first[q] ? (float)((double)p[q] / s_msum) : 0.0f;
  }
}

// Per-game commit, one CTA per game: children slot by slot against the running node count, then the backup of every
// LEAF slot.  The backup gathers one (node, slot, sign) entry per node of each LEAF path, sorts them by (node, slot) in
// shared memory and lets one thread add each node's entries in ascending slot order: the bits of a sequential
// slot-by-slot backup without a serial walk of L paths.  More entries than LB_ENTRIES (very deep paths) take that
// serial walk instead.  The same walks clear in_flight on every path of the batch.
constexpr int LB_THREADS = 256, LB_WARPS = LB_THREADS / 32;
constexpr int LB_ENTRIES = 4096;  // 32 KB of keys
static_assert(FPC_MAX_LEAVES_PER_GAME <= (1 << 30), "slot index and sign share the low 32 bits of a key");

template <class G>
__global__ void __launch_bounds__(LB_THREADS) leaves_commit_kernel(const fpc_tree T, const fpc_leaf_batch B, const float *values) {
  __shared__ unsigned long long s_ent[LB_ENTRIES];
  __shared__ int s_node[FPC_MAX_LEAVES_PER_GAME], s_cnt[FPC_MAX_LEAVES_PER_GAME], s_base[FPC_MAX_LEAVES_PER_GAME];
  __shared__ float s_val[FPC_MAX_LEAVES_PER_GAME];
  __shared__ int8_t s_what[FPC_MAX_LEAVES_PER_GAME];  // 0 no backup, 1 terminal LEAF, 2 LEAF in progress
  __shared__ int s_ne;
  const int g = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int L = B.L;
  const size_t s0 = (size_t)g * L, slab = (size_t)g * T.node_cap;
  if (tid == 0) s_ne = 0;
  for (int j = tid; j < L; j += LB_THREADS) {
    const int kind = B.slot_kind[s0 + j];
    const int result = B.leaf_status[s0 + j] & FPC_STATUS_RESULT_MASK;
    int what = 0;
    float v = 0.0f;
    if (kind == FPC_SLOT_LEAF) {
      what = result ? 1 : 2;
      v = result == 3 ? 0.0f : result ? -1.0f : values[s0 + j];
    }
    s_node[j] = kind == FPC_SLOT_EMPTY ? -1 : B.slot_node[s0 + j];
    s_what[j] = (int8_t)what;
    s_val[j] = v;
  }
  __syncthreads();
  // children per slot (one per non-zero prior), one warp per slot
  for (int j = warp; j < L; j += LB_WARPS) {
    int n = 0;
    if (s_what[j] == 2) {
      const int cnt = B.leaf_counts[s0 + j];
      for (int i0 = 0; i0 < cnt; i0 += 32) {
        const int i = i0 + lane;
        n += __popc(__ballot_sync(FULL, i < cnt && B.priors[(s0 + j) * MAX_MOVES + i] != 0.0f));
      }
    }
    if (lane == 0) s_cnt[j] = n;
  }
  __syncthreads();
  if (tid == 0) {  // allocation in slot order, each slot checked against the running count
    int nn = T.n_nodes[g], err = 0, drop = 0;
    for (int j = 0; j < L; ++j) {
      s_base[j] = -1;
      drop |= s_what[j] == 1;
      if (s_what[j] != 2) continue;
      if (nn + s_cnt[j] > T.node_cap) {
        err = ERR_NODE_CAP;
      } else {
        s_base[j] = nn;
        nn += s_cnt[j];
      }
    }
    T.n_nodes[g] = nn;
    if (err) T.error[g] |= err;
    if (drop) T.dropped[g] = 1;
  }
  __syncthreads();
  for (int j = warp; j < L; j += LB_WARPS) {
    const int base = s_base[j];
    if (base < 0) continue;
    const int leaf = s_node[j], cnt = B.leaf_counts[s0 + j];
    int written = 0;
    for (int i0 = 0; i0 < cnt; i0 += 32) {
      const int i = i0 + lane;
      const float prior = i < cnt ? B.priors[(s0 + j) * MAX_MOVES + i] : 0.0f;
      const bool make = i < cnt && prior != 0.0f;
      const unsigned bal = __ballot_sync(FULL, make);
      if (make) {
        const size_t c = slab + base + written + __popc(bal & ((1u << lane) - 1u));
        T.parent[c] = leaf;
        T.first_child[c] = 0;
        T.n_children[c] = 0;
        T.visits[c] = 1;  // node.h:28
        T.move_flat[c] = B.leaf_flat[(s0 + j) * MAX_MOVES + i];
        T.board_idx[c] = -1;
        T.value_sum[c] = 0.0;
        T.prior[c] = prior;
      }
      written += __popc(bal);
    }
    if (lane == 0) {
      T.first_child[slab + leaf] = base;
      T.n_children[slab + leaf] = s_cnt[j];
    }
  }
  // the paths, one thread per slot: clear the marks; gather the backup entries of the LEAF slots
  for (int j = tid; j < L; j += LB_THREADS) {
    const bool backup = s_what[j] != 0;
    unsigned par = 0;
    for (int node = s_node[j]; node >= 0; node = T.parent[slab + node], par ^= 1u) {
      B.in_flight[slab + node] = 0;
      if (backup) {
        const int e = atomicAdd(&s_ne, 1);
        if (e < LB_ENTRIES) s_ent[e] = (unsigned long long)node << 32 | (unsigned)j << 1 | par;
      }
    }
  }
  __syncthreads();
  const int ne = s_ne;
  if (ne > LB_ENTRIES) {  // Node::Backpropagate slot by slot
    if (tid == 0)
      for (int j = 0; j < L; ++j) {
        if (!s_what[j]) continue;
        double v = (double)s_val[j];
        for (int node = s_node[j]; node >= 0; node = T.parent[slab + node]) {
          T.value_sum[slab + node] += v;
          T.visits[slab + node] += 1;
          v = -v;
        }
      }
    return;
  }
  int np = 1;
  while (np < ne) np <<= 1;
  for (int e = ne + tid; e < np; e += LB_THREADS) s_ent[e] = ~0ull;
  __syncthreads();
  for (int kk = 2; kk <= np; kk <<= 1)  // bitonic sort, ascending
    for (int jj = kk >> 1; jj > 0; jj >>= 1) {
      for (int e = tid; e < np; e += LB_THREADS) {
        const int o = e ^ jj;
        if (o > e) {
          const unsigned long long a = s_ent[e], b = s_ent[o];
          if ((a > b) == ((e & kk) == 0)) {
            s_ent[e] = b;
            s_ent[o] = a;
          }
        }
      }
      __syncthreads();
    }
  for (int e = tid; e < ne; e += LB_THREADS) {
    const int node = (int)(s_ent[e] >> 32);
    if (e > 0 && (int)(s_ent[e - 1] >> 32) == node) continue;
    double acc = T.value_sum[slab + node];
    int n = 0;
    for (int t = e; t < ne && (int)(s_ent[t] >> 32) == node; ++t, ++n) {
      const unsigned lo = (unsigned)s_ent[t];
      const double v = (double)s_val[lo >> 1];
      acc += (lo & 1u) ? -v : v;
    }
    T.value_sum[slab + node] = acc;
    T.visits[slab + node] += n;
  }
}

// ---- Dirichlet noise on the root's children (fpc_tree_root_noise; the recipe is stated in include/fpc.h) ------------
constexpr int NOISE_ATTEMPTS = 64;  // Marsaglia-Tsang attempts before the deterministic fallback
constexpr double TWO_PI = 6.283185307179586;

// Uniform j of child i of the game with this key: never 0, so every log below is finite
__device__ __forceinline__ double noise_uniform(uint64_t seed, uint64_t key, int i, int j) {
  return ((double)(mix64(seed, key, (uint64_t)i << 32 | (uint32_t)j) >> 11) + 0.5) * 0x1p-53;
}

// Gamma(alpha, 1) for child i.  Attempt t reads uniforms 3t (Box-Muller radius), 3t+1 (angle) and 3t+2 (acceptance);
// the alpha < 1 boost reads uniform 3 * NOISE_ATTEMPTS, so the draws of a child never depend on which attempt accepted.
__device__ __noinline__ double noise_gamma(uint64_t seed, uint64_t key, int i, double alpha) {
  const double a = alpha < 1.0 ? alpha + 1.0 : alpha;
  const double d = a - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
  double g = d;
  for (int t = 0; t < NOISE_ATTEMPTS; ++t) {
    const double x = sqrt(-2.0 * log(noise_uniform(seed, key, i, 3 * t))) * cos(TWO_PI * noise_uniform(seed, key, i, 3 * t + 1));
    const double v = 1.0 + c * x;
    if (v <= 0.0) continue;
    const double v3 = v * v * v;
    if (log(noise_uniform(seed, key, i, 3 * t + 2)) < 0.5 * x * x + d - d * v3 + d * log(v3)) {
      g = d * v3;
      break;
    }
  }
  if (alpha < 1.0) g *= pow(noise_uniform(seed, key, i, 3 * NOISE_ATTEMPTS), 1.0 / alpha);
  return g;
}

// One warp per game, child i on lane i % 32: the draws, the f64 sum in a fixed order (lane-wise ascending i, then the
// xor tree), and the mix into the f32 priors.
__global__ void __launch_bounds__(SEL_WARPS * 32) tree_root_noise_kernel(const fpc_tree T, uint64_t seed, const int64_t *keys,
                                                                         double alpha, double eps, int32_t *done) {
  const int lane = threadIdx.x & 31;
  const int g = blockIdx.x * SEL_WARPS + (threadIdx.x >> 5);
  if (g >= T.n_games || done[g] || T.dropped[g]) return;
  const size_t slab = (size_t)g * T.node_cap;
  const int k = T.n_children[slab], fc = T.first_child[slab];
  if (k <= 0) return;
  const uint64_t key = (uint64_t)keys[g];
  constexpr int PER = (MAX_MOVES + 31) / 32;
  double gam[PER];
  double sum = 0.0;
#pragma unroll
  for (int q = 0; q < PER; ++q) {
    const int i = lane + 32 * q;
    gam[q] = i < k ? noise_gamma(seed, key, i, alpha) : 0.0;
    sum += gam[q];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(FULL, sum, o);
#pragma unroll
  for (int q = 0; q < PER; ++q) {
    const int i = lane + 32 * q;
    if (i < k) {
      const double eta = sum > 0.0 ? gam[q] / sum : 1.0 / k;  // sum 0: every draw underflowed (alpha below ~0.05)
      float *p = T.prior + slab + fc + i;
      *p = (float)((1.0 - eps) * (double)*p + eps * eta);
    }
  }
  if (lane == 0) done[g] = 1;
}

// ---- Gumbel root search (fpc_tree_select_gumbel / fpc_tree_gumbel_result; the semantics are stated in include/fpc.h) --
// One warp per game, root child i on lane i % 32 in register i / 32.  Every f64 sum runs lane-wise in ascending i, then
// over the xor butterfly 16 .. 1; products and sums are spelled __dmul_rn / __dadd_rn so that no FMA contraction changes
// the bits a restatement computes.
constexpr int GB_PER = (MAX_MOVES + 31) / 32;
constexpr int GUMBEL_J = INT32_MIN;  // the draws' uniform j = 2^31: a stream disjoint from the root noise's j <= 192
constexpr double GUMBEL_FLOOR = -1e9;

// mctx's get_sequence_of_considered_visits(m, n_sims)[s] in closed form, extended past n_sims.  Once c is 2 it stays 2,
// and every later phase adds one visit per two simulations.
__device__ __forceinline__ int considered_visits(int s, int m, int n_sims) {
  if (m <= 1) return s;
  int l2 = 0;
  while ((1 << l2) < m) ++l2;
  int c = m, v = 0;
  while (c > 2) {
    const int e = max(1, n_sims / (l2 * c));
    if (s < e * c) return v + s / c;
    s -= e * c;
    v += e;
    c = max(2, c / 2);
  }
  return v + s / 2;
}

// The root's network value u: value_sum[0] when s == 0, else root_value[g]; the select (write) records it as
// root_value when s == 0.
struct RootValue {
  const fpc_tree &T;
  const fpc_gumbel &B;
  int g, lane;
  bool write;
  __device__ __forceinline__ double operator()(int s, size_t slab) const {
    const double root = s == 0 ? T.value_sum[slab] : B.root_value[g];
    if (write && s == 0 && lane == 0) B.root_value[g] = root;
    return root;
  }
};

// Game g's node with k > 0 children (the first at fc): n = N_i and z = l_i + sigma_i in this lane's registers,
// nmax = max N_i; returns s = sum N_i.  value(s, slab) is the node's network value u (v = -u), which the caller reads,
// and caches when s == 0: RootValue at the root, node_value below it.  With in_flight (a leaf batch's marks, slab of
// game g) the statistics are the effective ones, N_i + VL*in_flight and W_i - VL*in_flight, while value() still receives
// the committed s.
template <class Value>
__device__ __forceinline__ int gumbel_logits(const fpc_tree &T, const fpc_gumbel &B, int g, int lane, int fc, int k,
                                             Value value, int (&n)[GB_PER], double (&z)[GB_PER], int &nmax,
                                             const int32_t *in_flight = nullptr, int VL = 0) {
  const size_t slab = (size_t)g * T.node_cap;
  double q[GB_PER];
  int s = 0, s_committed = 0;
  nmax = INT32_MIN;
  double lmax = -CUDART_INF, wq = 0.0, ws = 0.0;
#pragma unroll
  for (int r = 0; r < GB_PER; ++r) {
    const int i = lane + 32 * r;
    n[r] = -1, q[r] = 0.0;
    if (i < k) {
      const size_t c = slab + fc + i;
      const double p = (double)T.prior[c];
      const int vl = in_flight ? VL * in_flight[fc + i] : 0;
      n[r] = T.visits[c] - 1;  // children are created with visit_count 1 (node.h:28)
      if (in_flight) s_committed += n[r], n[r] += vl;
      lmax = fmax(lmax, log(p));
      s += n[r];
      nmax = max(nmax, n[r]);
      if (n[r] > 0) {
        q[r] = (in_flight ? T.value_sum[c] - (double)vl : T.value_sum[c]) / (double)n[r];
        const double w = fmax(p, 0x1p-126);
        wq = __dadd_rn(wq, __dmul_rn(w, q[r]));
        ws = __dadd_rn(ws, w);
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(FULL, s, o);
    if (in_flight) s_committed += __shfl_xor_sync(FULL, s_committed, o);
    nmax = max(nmax, __shfl_xor_sync(FULL, nmax, o));
    lmax = fmax(lmax, __shfl_xor_sync(FULL, lmax, o));
    wq = __dadd_rn(wq, __shfl_xor_sync(FULL, wq, o));
    ws = __dadd_rn(ws, __shfl_xor_sync(FULL, ws, o));
  }
  const double root = value(in_flight ? s_committed : s, slab);
  const double w_mean = ws > 0.0 ? wq / ws : 0.0;
  const double v_mix = __dadd_rn(-root, __dmul_rn((double)s, w_mean)) / (1.0 + (double)s);
  double lo = CUDART_INF, hi = -CUDART_INF;
#pragma unroll
  for (int r = 0; r < GB_PER; ++r) {
    if (lane + 32 * r < k) {
      if (n[r] <= 0) q[r] = v_mix;  // completed Q
      lo = fmin(lo, q[r]);
      hi = fmax(hi, q[r]);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = fmin(lo, __shfl_xor_sync(FULL, lo, o));
    hi = fmax(hi, __shfl_xor_sync(FULL, hi, o));
  }
  const double span = fmax(hi - lo, 1e-8);
  const double a = __dmul_rn(B.c_visit + (double)nmax, B.c_scale);
  // log p_i is taken again here rather than kept in registers across the divisions above
#pragma unroll
  for (int r = 0; r < GB_PER; ++r) {
    const int i = lane + 32 * r;
    z[r] = i < k ? __dadd_rn(log((double)T.prior[slab + fc + i]) - lmax, __dmul_rn(a, (q[r] - lo) / span)) : -CUDART_INF;
  }
  return s;
}

// The child index maximising max(GUMBEL_FLOOR, g_i + z_i) over the children with N_i == cv (the first maximum in
// ascending i), or -1 when there is none.
__device__ __forceinline__ int gumbel_argmax(const fpc_gumbel &B, uint64_t key, int lane, int k, int cv,
                                             const int (&n)[GB_PER], const double (&z)[GB_PER]) {
  double best = -CUDART_INF;
  int best_i = 0x7fffffff;
#pragma unroll
  for (int r = 0; r < GB_PER; ++r) {
    const int i = lane + 32 * r;
    if (i < k && n[r] == cv) {
      const double gum = -log(-log(noise_uniform(B.seed, key, i, GUMBEL_J)));
      const double x = __dadd_rn(__dmul_rn(B.scale, gum), z[r]);
      const double score = x > GUMBEL_FLOOR ? x : GUMBEL_FLOOR;
      if (score > best) {  // strict: the first maximum wins
        best = score;
        best_i = i;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ob = __shfl_xor_sync(FULL, best, o);
    const int oi = __shfl_xor_sync(FULL, best_i, o);
    if (oi != 0x7fffffff && (best_i == 0x7fffffff || ob > best || (ob == best && oi < best_i))) {
      best = ob;
      best_i = oi;
    }
  }
  return best_i == 0x7fffffff ? -1 : best_i;
}

// The Gumbel root step (descend's root_step): the root's child by sequential halving.
__device__ __forceinline__ bool gumbel_root_step(const fpc_tree &T, const fpc_gumbel &B, int g, int lane, int &node,
                                                 int &nc, int &fc, int &nv) {
  if (nc <= 0) return true;  // an unexpanded root is the leaf, as in fpc_tree_select
  int n[GB_PER], nmax;
  double z[GB_PER];
  const int s = gumbel_logits(T, B, g, lane, fc, nc, RootValue{T, B, g, lane, true}, n, z, nmax);
  const int i = gumbel_argmax(B, (uint64_t)B.keys[g], lane, nc, considered_visits(s, min(B.max_considered, nc), B.n_sims), n, z);
  if (i < 0) {  // a root visit left the schedule: drop the game as a failed SelectChild does
    if (lane == 0) {
      T.error[g] |= ERR_NO_CHILD;
      T.leaf[g] = -1;
      T.dropped[g] = 1;
    }
    return false;
  }
  const size_t slab = (size_t)g * T.node_cap;
  node = fc + i;
  nc = T.n_children[slab + node], fc = T.first_child[slab + node], nv = T.visits[slab + node];
  return true;
}

// e_i = exp(z_i - max_j z_j) in place of z (0 for i >= k); returns E = sum e_i, both in the stated order.
__device__ __forceinline__ double softmax_terms(int lane, int k, double (&z)[GB_PER]) {
  double zmax = -CUDART_INF, sum = 0.0;
#pragma unroll
  for (int r = 0; r < GB_PER; ++r)
    if (lane + 32 * r < k) zmax = fmax(zmax, z[r]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) zmax = fmax(zmax, __shfl_xor_sync(FULL, zmax, o));
#pragma unroll
  for (int r = 0; r < GB_PER; ++r) {
    z[r] = lane + 32 * r < k ? exp(z[r] - zmax) : 0.0;
    sum = __dadd_rn(sum, z[r]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum = __dadd_rn(sum, __shfl_xor_sync(FULL, sum, o));
  return sum;
}

// Gumbel MuZero's interior step at node x of game g (k > 0 children, the first at fc): the index of the first maximum of
// pi'_i - N_i / (1 + s), or -1 when no score compares greater than -inf.  x's network value is value_sum[x] when the
// committed s is 0 (then cached in cache[x]), else cache[x]; both are requested in the children's memory round.  With
// in_flight the statistics are a leaf batch's effective ones (gumbel_logits).
__device__ __forceinline__ int interior_argmax(const fpc_tree &T, const fpc_gumbel &B, int g, int lane, int x, int fc, int k,
                                               double *cache, const int32_t *in_flight = nullptr, int VL = 0) {
  const size_t slab = (size_t)g * T.node_cap;
  const double own = T.value_sum[slab + x], cached = cache[x];
  int n[GB_PER], nmax;
  double z[GB_PER];
  const int s = gumbel_logits(T, B, g, lane, fc, k,
                              [&](int s, size_t) {
                                if (s == 0 && lane == 0) cache[x] = own;
                                return s == 0 ? own : cached;
                              },
                              n, z, nmax, in_flight, VL);
  const double E = softmax_terms(lane, k, z);
  const double d = 1.0 + (double)s;
  double best = -CUDART_INF;
  int best_i = 0x7fffffff;
#pragma unroll
  for (int r = 0; r < GB_PER; ++r) {
    const int i = lane + 32 * r;
    if (i < k) {
      const double score = __dsub_rn(z[r] / E, (double)n[r] / d);
      if (score > best) {  // strict: the first maximum wins
        best = score;
        best_i = i;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ob = __shfl_xor_sync(FULL, best, o);
    const int oi = __shfl_xor_sync(FULL, best_i, o);
    if (oi != 0x7fffffff && (best_i == 0x7fffffff || ob > best || (ob == best && oi < best_i))) {
      best = ob;
      best_i = oi;
    }
  }
  return best_i == 0x7fffffff ? -1 : best_i;
}

// fpc_tree_select with the Gumbel root step: the root's child by sequential halving, then Node::SelectChild below it.
template <class G>
__global__ void __launch_bounds__(SEL_WARPS * 32) tree_descend_gumbel_kernel(const fpc_tree T, const fpc_gumbel B) {
  __shared__ alignas(16) uint8_t recs[SEL_WARPS][256];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * SEL_WARPS + wib;
  if (g >= T.n_games) return;
  if (T.dropped[g]) {
    if (lane == 0) T.leaf[g] = -1;
    return;
  }
  descend<G>(T, g, lane, recs[wib],
             [&](int &node, int &nc, int &fc, int &nv) { return gumbel_root_step(T, B, g, lane, node, nc, fc, nv); });
}

// fpc_tree_select with the Gumbel root step and Gumbel MuZero's interior step below it: at node x the child maximising
// pi'_i - N_i / (1 + s), pi' = softmax(l + sigma(completed Q)) with x's own network value, cached in node_value[x] the
// first time the descent passes x (s == 0).  x's value_sum and node_value are requested in the children's memory
// round; the winner's child range is loaded after the arg-max.
template <class G>
__global__ void __launch_bounds__(SEL_WARPS * 32) tree_descend_gumbel_interior_kernel(const fpc_tree T, const fpc_gumbel B,
                                                                                       double *node_value) {
  __shared__ alignas(16) uint8_t recs[SEL_WARPS][256];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * SEL_WARPS + wib;
  if (g >= T.n_games) return;
  if (T.dropped[g]) {
    if (lane == 0) T.leaf[g] = -1;
    return;
  }
  const size_t slab = (size_t)g * T.node_cap;
  double *cache = node_value + slab;
  descend<G>(
      T, g, lane, recs[wib],
      [&](int &node, int &nc, int &fc, int &nv) { return gumbel_root_step(T, B, g, lane, node, nc, fc, nv); },
      [&](int &node, int &nc, int &fc, int &) {  // nv (SelectChild's parent count) is not used below the root
        const int i = interior_argmax(T, B, g, lane, node, fc, nc, cache);
        if (i < 0) {  // NaN scores
          if (lane == 0) {
            T.error[g] |= ERR_NO_CHILD;
            T.leaf[g] = -1;
            T.dropped[g] = 1;
          }
          return false;
        }
        node = fc + i;
        nc = T.n_children[slab + node], fc = T.first_child[slab + node];
        return true;
      });
}

// ---- leaf-parallel Gumbel search (fpc_tree_select_gumbel_leaves / fpc_tree_gumbel_result_leaves; include/fpc.h) ----
// One warp per game, its L slots in order through leaves_select.  The root's scores come from the committed statistics
// once per batch (gumbel_logits and the draws: one reduction per game and batch); the schedule runs on issued[] (I_i in
// register i / 32 of lane i % 32), so slot j's root child is the first maximum of score_i over {I_i == cv(sum I)}.  Below
// it the descent is leaves_select's SelectChild with virtual loss, or with Interior the interior step over the effective
// statistics.  A slot whose descent fails after its root step gives its issue back: only LEAF and COLLISION slots count.
template <class G, bool Interior>
__global__ void __launch_bounds__(SEL_WARPS * 32) gumbel_leaves_descend_kernel(const fpc_tree T, const fpc_gumbel Gb,
                                                                              const fpc_leaf_batch B, int32_t *issued,
                                                                              double *node_value) {
  __shared__ alignas(16) uint8_t recs[SEL_WARPS][256];
  __shared__ int paths[SEL_WARPS][LB_PATH];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * SEL_WARPS + wib;
  if (g >= T.n_games) return;
  const size_t slab = (size_t)g * T.node_cap;
  const int k = T.n_children[slab], fc0 = T.first_child[slab];
  const bool root_open = !T.dropped[g] && k > 0;
  int32_t *iss = issued + (size_t)g * MAX_MOVES;
  const int32_t *in_flight = B.in_flight + slab;
  int I[GB_PER];
  double score[GB_PER];
  int t = 0, mp = 0;
  if (root_open) {
    int n[GB_PER], nmax;
    double z[GB_PER];
    gumbel_logits(T, Gb, g, lane, fc0, k, RootValue{T, Gb, g, lane, true}, n, z, nmax);
    const uint64_t key = (uint64_t)Gb.keys[g];
#pragma unroll
    for (int r = 0; r < GB_PER; ++r) {
      const int i = lane + 32 * r;
      I[r] = i < k ? iss[i] : 0;
      t += I[r];
      score[r] = -CUDART_INF;
      if (i < k) {  // gumbel_argmax's score
        const double gum = -log(-log(noise_uniform(Gb.seed, key, i, GUMBEL_J)));
        const double x = __dadd_rn(__dmul_rn(Gb.scale, gum), z[r]);
        score[r] = x > GUMBEL_FLOOR ? x : GUMBEL_FLOOR;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(FULL, t, o);
    mp = min(Gb.max_considered, k);
  }
  int taken = 0, last = -1;
  auto root_step = [&](int &node, int &depth, int &nc, int &fc, int &nv) -> int {
    if (nc <= 0) return 0;  // an unexpanded root is every slot's endpoint: one LEAF, L - 1 COLLISIONs
    const int cv = considered_visits(t, mp, Gb.n_sims);
    double best = -CUDART_INF;
    int best_i = 0x7fffffff;
#pragma unroll
    for (int r = 0; r < GB_PER; ++r) {
      const int i = lane + 32 * r;
      if (i < k && I[r] == cv && score[r] > best) {  // strict: the first maximum wins
        best = score[r];
        best_i = i;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ob = __shfl_xor_sync(FULL, best, o);
      const int oi = __shfl_xor_sync(FULL, best_i, o);
      if (oi != 0x7fffffff && (best_i == 0x7fffffff || ob > best || (ob == best && oi < best_i))) {
        best = ob;
        best_i = oi;
      }
    }
    if (best_i == 0x7fffffff) return ERR_NO_CHILD;  // a root visit left the schedule
#pragma unroll
    for (int r = 0; r < GB_PER; ++r) I[r] += lane + 32 * r == best_i;
    ++t, ++taken, last = best_i;
    node = fc + best_i;
    depth = 1;
    if (lane == 0) paths[wib][1] = node;
    nc = T.n_children[slab + node], fc = T.first_child[slab + node];
    nv = T.visits[slab + node] + B.virtual_loss * in_flight[node];
    return 0;
  };
  int filled;
  if constexpr (Interior) {
    double *cache = node_value + slab;
    filled = leaves_select<G>(T, B, g, lane, recs[wib], paths[wib], root_step, [&](int node, int nc, int fc) {
      return interior_argmax(T, Gb, g, lane, node, fc, nc, cache, in_flight, B.virtual_loss);
    });
  } else {
    filled = leaves_select<G>(T, B, g, lane, recs[wib], paths[wib], root_step);
  }
  if (!root_open) return;
  if (taken > filled) {  // the slot that failed below its root step is EMPTY: it issued no visit
#pragma unroll
    for (int r = 0; r < GB_PER; ++r) I[r] -= lane + 32 * r == last;
  }
#pragma unroll
  for (int r = 0; r < GB_PER; ++r)
    if (lane + 32 * r < k) iss[lane + 32 * r] = I[r];
}

// The action (the considered child at cv = Nmax with the best score) and the improved policy softmax(l + sigma).  With
// issued (a leaf-parallel search's I_i) the survivors are {I_i == max I} instead.
__device__ __forceinline__ void gumbel_result(const fpc_tree &T, const fpc_gumbel &B, int g, int lane, const int32_t *issued,
                                              int32_t *action, float *policy) {
  const size_t slab = (size_t)g * T.node_cap;
  const int k = T.n_children[slab], fc = T.first_child[slab];
  float *row = policy + (size_t)g * MAX_MOVES;
  if (k <= 0) {
    for (int i = lane; i < MAX_MOVES; i += 32) row[i] = 0.0f;
    if (lane == 0) action[g] = -1;
    return;
  }
  int n[GB_PER], nmax;
  double z[GB_PER];
  gumbel_logits(T, B, g, lane, fc, k, RootValue{T, B, g, lane, false}, n, z, nmax);
  if (issued) {
    nmax = INT32_MIN;
#pragma unroll
    for (int r = 0; r < GB_PER; ++r) {
      const int i = lane + 32 * r;
      n[r] = i < k ? issued[(size_t)g * MAX_MOVES + i] : -1;
      nmax = max(nmax, n[r]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) nmax = max(nmax, __shfl_xor_sync(FULL, nmax, o));
  }
  const int best = gumbel_argmax(B, (uint64_t)B.keys[g], lane, k, nmax, n, z);
  const double sum = softmax_terms(lane, k, z);
#pragma unroll
  for (int r = 0; r < GB_PER; ++r) {
    const int i = lane + 32 * r;
    if (i < MAX_MOVES) row[i] = (float)(z[r] / sum);
  }
  if (lane == 0) action[g] = best < 0 ? -1 : T.move_flat[slab + fc + best];
}

__global__ void __launch_bounds__(SEL_WARPS * 32) tree_gumbel_result_kernel(const fpc_tree T, const fpc_gumbel B,
                                                                             int32_t *action, float *policy) {
  const int g = blockIdx.x * SEL_WARPS + (threadIdx.x >> 5);
  if (g >= T.n_games) return;
  gumbel_result(T, B, g, threadIdx.x & 31, nullptr, action, policy);
}

__global__ void __launch_bounds__(SEL_WARPS * 32) tree_gumbel_result_leaves_kernel(const fpc_tree T, const fpc_gumbel B,
                                                                                    const int32_t *issued, int32_t *action,
                                                                                    float *policy) {
  const int g = blockIdx.x * SEL_WARPS + (threadIdx.x >> 5);
  if (g >= T.n_games) return;
  gumbel_result(T, B, g, threadIdx.x & 31, issued, action, policy);
}

// ---- Keyed move sampling from the root's visit counts (fpc_tree_sample_root; the recipe is stated in include/fpc.h) --
constexpr int SAMPLE_J = INT32_MIN + 1;  // uniform j = 2^31 + 1: disjoint from the root noise's j <= 192 and Gumbel's 2^31

// One warp per game: the lanes compute the weights of children i = lane, lane + 32, ... into shared memory, then lane 0
// runs the prefix sum in ascending i (the one order the header states) and picks the child.
__global__ void __launch_bounds__(SEL_WARPS * 32) tree_sample_root_kernel(const fpc_tree T, uint64_t seed, const int64_t *keys,
                                                                           double temperature, int32_t *action) {
  __shared__ double s_w[SEL_WARPS][MAX_MOVES];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = blockIdx.x * SEL_WARPS + warp;
  if (g >= T.n_games) return;
  const size_t slab = (size_t)g * T.node_cap;
  const int k = T.dropped[g] ? 0 : min(T.n_children[slab], MAX_MOVES);
  if (k <= 0) {
    if (lane == 0) action[g] = -1;
    return;
  }
  const int fc = T.first_child[slab];
  long long vsum = 0;
  for (int i = lane; i < k; i += 32) vsum += max(T.visits[slab + fc + i], 0);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) vsum += __shfl_xor_sync(FULL, vsum, o);
  const double V = (double)vsum, inv_t = 1.0 / temperature;
  for (int i = lane; i < k; i += 32) {
    const double v = (double)max(T.visits[slab + fc + i], 0);
    s_w[warp][i] = temperature == 1.0 ? v : pow(v / V, inv_t);
  }
  __syncwarp();
  if (lane != 0) return;
  double W = 0.0;
  int last = -1;
  for (int i = 0; i < k; ++i) {
    W = __dadd_rn(W, s_w[warp][i]);
    if (s_w[warp][i] > 0.0) last = i;
  }
  if (!(W > 0.0)) {  // no visits, or every weight underflowed
    action[g] = -1;
    return;
  }
  const double u = __dmul_rn(noise_uniform(seed, (uint64_t)keys[g], 0, SAMPLE_J), W);
  int pick = last;  // U*W rounded up to W: the last child with weight
  double P = 0.0;
  for (int i = 0; i < k; ++i) {
    P = __dadd_rn(P, s_w[warp][i]);
    if (P > u) {
      pick = i;
      break;
    }
  }
  action[g] = T.move_flat[slab + fc + pick];
}

static int check_tree(const fpc_tree *t, const char *who) {
  if (!t) return fail(FPC_ERR_ARG, std::string(who) + ": null tree");
  if (!fpc_supported(t->R) || t->n_games < 0 || t->node_cap < 1 || t->board_cap < 1)
    return fail(FPC_ERR_ARG, std::string(who) + ": bad tree geometry");
  if (t->n_games > 0 &&
      (!t->parent || !t->first_child || !t->n_children || !t->visits || !t->move_flat || !t->board_idx ||
       !t->value_sum || !t->prior || !t->n_nodes || !t->n_boards || !t->leaf || !t->dropped || !t->error ||
       !t->boards || !t->leaf_boards || !t->leaf_flat || !t->leaf_counts || !t->leaf_status || !t->k))
    return fail(FPC_ERR_ARG, std::string(who) + ": null tree array");
  return FPC_OK;
}

static int check_batch(const fpc_tree *t, const fpc_leaf_batch *b, const char *who) {
  if (!b) return fail(FPC_ERR_ARG, std::string(who) + ": null leaf batch");
  if (b->L < 1 || b->L > FPC_MAX_LEAVES_PER_GAME)
    return fail(FPC_ERR_ARG, std::string(who) + ": L = " + std::to_string(b->L) + " outside 1 .. " +
                                 std::to_string(FPC_MAX_LEAVES_PER_GAME));
  if (b->virtual_loss < 1) return fail(FPC_ERR_ARG, std::string(who) + ": virtual_loss below 1");
  if ((int64_t)t->n_games * b->L > INT32_MAX) return fail(FPC_ERR_ARG, std::string(who) + ": n_games * L too large");
  if (t->n_games > 0 && (!b->in_flight || !b->slot_node || !b->slot_kind || !b->leaf_boards || !b->leaf_flat ||
                         !b->leaf_counts || !b->leaf_status || !b->k || !b->priors || !b->collisions))
    return fail(FPC_ERR_ARG, std::string(who) + ": null leaf-batch array");
  return FPC_OK;
}

template <class G>
static int launch_advance(const fpc_tree &t, const int32_t *actions, const uint8_t *roots, int max_nodes, int max_boards,
                          int32_t *kept, cudaStream_t st) {
  const size_t smem = 2 * sizeof(uint32_t) * (size_t)((t.node_cap + 31) / 32);
  if (smem > 48 * 1024)
    CK(cudaFuncSetAttribute(tree_advance_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  tree_advance_kernel<G><<<t.n_games, ADV_THREADS, smem, st>>>(t, actions, roots, max_nodes, max_boards, kept);
  return cuda_check(cudaGetLastError(), "tree_advance_kernel launch");
}

static int check_gumbel(const fpc_tree *t, const fpc_gumbel *gb, const char *who) {
  if (!gb) return fail(FPC_ERR_ARG, std::string(who) + ": null gumbel");
  if (gb->max_considered < 1 || gb->max_considered > FPC_MAX_MOVES)
    return fail(FPC_ERR_ARG, std::string(who) + ": max_considered " + std::to_string(gb->max_considered) + " outside 1 .. " +
                                 std::to_string(FPC_MAX_MOVES));
  if (gb->n_sims < 0) return fail(FPC_ERR_ARG, std::string(who) + ": negative n_sims");
  const double params[3] = {gb->scale, gb->c_visit, gb->c_scale};
  const char *names[3] = {"scale", "c_visit", "c_scale"};
  for (int i = 0; i < 3; ++i)
    if (!(params[i] >= 0.0) || !std::isfinite(params[i]))
      return fail(FPC_ERR_ARG, std::string(who) + ": " + names[i] + " must be non-negative and finite");
  if (t->n_games > 0 && (!gb->keys || !gb->root_value)) return fail(FPC_ERR_ARG, std::string(who) + ": null keys / root_value");
  return FPC_OK;
}

// What fpc_tree_select does after its descent: the rules kernel on the leaf batch (legal moves + GetGameResult) and the
// planes, rotated by the first live leaf's colour with batch_rotation.
static int observe_leaves(const fpc_tree *t, int batch_rotation, float *d_planes, int flags, fpc_dense_track *track,
                          void *stream) {
  if (batch_rotation) {
    // the batch rotation is that of the first NON-terminal leaf: results first, then k, then the planes
    int rc = fpc_observe(t->R, t->leaf_boards, t->n_games, nullptr, t->leaf_flat, t->leaf_counts, t->leaf_status, nullptr,
                         nullptr, 0, nullptr, 0, stream);
    if (rc != FPC_OK) return rc;
    rc = dispatch(t->R, [&](auto g) {
      tree_batch_k_kernel<decltype(g)><<<1, 1024, 0, (cudaStream_t)stream>>>(*t);
      return cuda_check(cudaGetLastError(), "tree_batch_k_kernel launch");
    });
    if (rc != FPC_OK) return rc;
    return fpc_observe_tracked(track, t->R, t->leaf_boards, t->n_games, nullptr, nullptr, nullptr, nullptr, d_planes, t->k, 0,
                               nullptr, flags, stream);
  }
  // legal moves + GetGameResult + planes of the leaf batch: the environment's rules kernel
  return fpc_observe_tracked(track, t->R, t->leaf_boards, t->n_games, nullptr, t->leaf_flat, t->leaf_counts, t->leaf_status,
                             d_planes, t->k, 0, nullptr, flags, stream);
}

// What fpc_tree_select_leaves does after its selection: the rules kernel on the slots and their planes, rotated by the
// first LEAF slot in progress with batch_rotation.
static int observe_slots(const fpc_tree *t, const fpc_leaf_batch *b, int batch_rotation, float *d_planes, int flags,
                         fpc_dense_track *track, void *stream) {
  const int n_slots = t->n_games * b->L;
  if (batch_rotation) {
    int rc = fpc_observe(t->R, b->leaf_boards, n_slots, nullptr, b->leaf_flat, b->leaf_counts, b->leaf_status, nullptr,
                         nullptr, 0, nullptr, 0, stream);
    if (rc != FPC_OK) return rc;
    rc = dispatch(t->R, [&](auto g) {
      leaves_batch_k_kernel<decltype(g)><<<1, 1024, 0, (cudaStream_t)stream>>>(*b, n_slots);
      return cuda_check(cudaGetLastError(), "leaves_batch_k_kernel launch");
    });
    if (rc != FPC_OK) return rc;
    return fpc_observe_tracked(track, t->R, b->leaf_boards, n_slots, nullptr, nullptr, nullptr, nullptr, d_planes, b->k, 0,
                               nullptr, flags, stream);
  }
  return fpc_observe_tracked(track, t->R, b->leaf_boards, n_slots, nullptr, b->leaf_flat, b->leaf_counts, b->leaf_status,
                             d_planes, b->k, 0, nullptr, flags, stream);
}

}  // namespace fpc

using namespace fpc;

extern "C" {

int fpc_tree_reset(const fpc_tree *t, const uint8_t *d_root_boards, void *stream) {
  int rc = check_tree(t, "fpc_tree_reset");
  if (rc != FPC_OK) return rc;
  if (t->n_games == 0) return FPC_OK;
  if (!d_root_boards) return fail(FPC_ERR_ARG, "fpc_tree_reset: null roots");
  cudaStream_t st = (cudaStream_t)stream;
  return dispatch(t->R, [&](auto g) {
    tree_reset_kernel<decltype(g)><<<t->n_games, 256, 0, st>>>(*t, d_root_boards);
    return cuda_check(cudaGetLastError(), "tree_reset_kernel launch");
  });
}

int fpc_tree_advance(const fpc_tree *t, const int32_t *d_actions, const uint8_t *d_root_boards, int32_t max_keep_nodes,
                     int32_t max_keep_boards, int32_t *d_kept, void *stream) {
  int rc = check_tree(t, "fpc_tree_advance");
  if (rc != FPC_OK) return rc;
  if (t->node_cap > FPC_TREE_ADVANCE_MAX_NODE_CAP)
    return fail(FPC_ERR_ARG, "fpc_tree_advance: node_cap " + std::to_string(t->node_cap) + " above " +
                                 std::to_string(FPC_TREE_ADVANCE_MAX_NODE_CAP));
  if (max_keep_nodes < 0 || max_keep_boards < 0) return fail(FPC_ERR_ARG, "fpc_tree_advance: negative limit");
  if (t->n_games == 0) return FPC_OK;
  if (!d_actions || !d_root_boards) return fail(FPC_ERR_ARG, "fpc_tree_advance: null actions / roots");
  if (reinterpret_cast<uintptr_t>(d_root_boards) & 15) return fail(FPC_ERR_ARG, "root boards must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  return dispatch(t->R, [&](auto g) {
    return launch_advance<decltype(g)>(*t, d_actions, d_root_boards, max_keep_nodes, max_keep_boards, d_kept, st);
  });
}

int fpc_tree_select(const fpc_tree *t, int batch_rotation, float *d_planes, int flags, fpc_dense_track *track, void *stream) {
  int rc = check_tree(t, "fpc_tree_select");
  if (rc != FPC_OK) return rc;
  if (t->n_games == 0) return FPC_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = (t->n_games + SEL_WARPS - 1) / SEL_WARPS;
  rc = dispatch(t->R, [&](auto g) {
    tree_descend_kernel<decltype(g)><<<blocks, SEL_WARPS * 32, 0, st>>>(*t);
    return cuda_check(cudaGetLastError(), "tree_descend_kernel launch");
  });
  if (rc != FPC_OK) return rc;
  return observe_leaves(t, batch_rotation, d_planes, flags, track, stream);
}

int fpc_tree_select_gumbel(const fpc_tree *t, const fpc_gumbel *gb, int batch_rotation, float *d_planes, int flags,
                           fpc_dense_track *track, void *stream) {
  int rc = check_tree(t, "fpc_tree_select_gumbel");
  if (rc == FPC_OK) rc = check_gumbel(t, gb, "fpc_tree_select_gumbel");
  if (rc != FPC_OK) return rc;
  if (t->n_games == 0) return FPC_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = (t->n_games + SEL_WARPS - 1) / SEL_WARPS;
  rc = dispatch(t->R, [&](auto g) {
    tree_descend_gumbel_kernel<decltype(g)><<<blocks, SEL_WARPS * 32, 0, st>>>(*t, *gb);
    return cuda_check(cudaGetLastError(), "tree_descend_gumbel_kernel launch");
  });
  if (rc != FPC_OK) return rc;
  return observe_leaves(t, batch_rotation, d_planes, flags, track, stream);
}

int fpc_tree_select_gumbel_interior(const fpc_tree *t, const fpc_gumbel *gb, double *d_node_value, int batch_rotation,
                                    float *d_planes, int flags, fpc_dense_track *track, void *stream) {
  int rc = check_tree(t, "fpc_tree_select_gumbel_interior");
  if (rc == FPC_OK) rc = check_gumbel(t, gb, "fpc_tree_select_gumbel_interior");
  if (rc != FPC_OK) return rc;
  if (!d_node_value) return fail(FPC_ERR_ARG, "fpc_tree_select_gumbel_interior: null node_value");
  if (t->n_games == 0) return FPC_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = (t->n_games + SEL_WARPS - 1) / SEL_WARPS;
  rc = dispatch(t->R, [&](auto g) {
    tree_descend_gumbel_interior_kernel<decltype(g)><<<blocks, SEL_WARPS * 32, 0, st>>>(*t, *gb, d_node_value);
    return cuda_check(cudaGetLastError(), "tree_descend_gumbel_interior_kernel launch");
  });
  if (rc != FPC_OK) return rc;
  return observe_leaves(t, batch_rotation, d_planes, flags, track, stream);
}

int fpc_tree_gumbel_result(const fpc_tree *t, const fpc_gumbel *gb, int32_t *d_action, float *d_policy, void *stream) {
  int rc = check_tree(t, "fpc_tree_gumbel_result");
  if (rc == FPC_OK) rc = check_gumbel(t, gb, "fpc_tree_gumbel_result");
  if (rc != FPC_OK) return rc;
  if (t->n_games == 0) return FPC_OK;
  if (!d_action || !d_policy) return fail(FPC_ERR_ARG, "fpc_tree_gumbel_result: null action / policy");
  const int blocks = (t->n_games + SEL_WARPS - 1) / SEL_WARPS;
  tree_gumbel_result_kernel<<<blocks, SEL_WARPS * 32, 0, (cudaStream_t)stream>>>(*t, *gb, d_action, d_policy);
  return cuda_check(cudaGetLastError(), "tree_gumbel_result_kernel launch");
}

int fpc_tree_expand_backup(const fpc_tree *t, const float *d_logits, const float *d_values, void *stream) {
  int rc = check_tree(t, "fpc_tree_expand_backup");
  if (rc != FPC_OK) return rc;
  if (t->n_games == 0) return FPC_OK;
  if (!d_logits || !d_values) return fail(FPC_ERR_ARG, "fpc_tree_expand_backup: null logits / values");
  if (reinterpret_cast<uintptr_t>(d_logits) & 15) return fail(FPC_ERR_ARG, "logits must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  return dispatch(t->R, [&](auto g) {
    tree_expand_backup_kernel<decltype(g)><<<t->n_games, EXP_THREADS, 0, st>>>(*t, d_logits, d_values);
    return cuda_check(cudaGetLastError(), "tree_expand_backup_kernel launch");
  });
}

int fpc_tree_select_leaves(const fpc_tree *t, const fpc_leaf_batch *b, int batch_rotation, float *d_planes, int flags,
                           fpc_dense_track *track, void *stream) {
  int rc = check_tree(t, "fpc_tree_select_leaves");
  if (rc == FPC_OK) rc = check_batch(t, b, "fpc_tree_select_leaves");
  if (rc != FPC_OK) return rc;
  if (t->n_games == 0) return FPC_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = (t->n_games + SEL_WARPS - 1) / SEL_WARPS;
  rc = dispatch(t->R, [&](auto g) {
    leaves_descend_kernel<decltype(g)><<<blocks, SEL_WARPS * 32, 0, st>>>(*t, *b);
    return cuda_check(cudaGetLastError(), "leaves_descend_kernel launch");
  });
  if (rc != FPC_OK) return rc;
  return observe_slots(t, b, batch_rotation, d_planes, flags, track, stream);
}

int fpc_tree_select_gumbel_leaves(const fpc_tree *t, const fpc_gumbel *gb, const fpc_leaf_batch *b, int32_t *d_issued,
                                  double *d_node_value, int batch_rotation, float *d_planes, int flags,
                                  fpc_dense_track *track, void *stream) {
  int rc = check_tree(t, "fpc_tree_select_gumbel_leaves");
  if (rc == FPC_OK) rc = check_gumbel(t, gb, "fpc_tree_select_gumbel_leaves");
  if (rc == FPC_OK) rc = check_batch(t, b, "fpc_tree_select_gumbel_leaves");
  if (rc != FPC_OK) return rc;
  if (t->n_games == 0) return FPC_OK;
  if (!d_issued) return fail(FPC_ERR_ARG, "fpc_tree_select_gumbel_leaves: null issued");
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = (t->n_games + SEL_WARPS - 1) / SEL_WARPS;
  rc = dispatch(t->R, [&](auto g) {
    if (d_node_value)
      gumbel_leaves_descend_kernel<decltype(g), true><<<blocks, SEL_WARPS * 32, 0, st>>>(*t, *gb, *b, d_issued, d_node_value);
    else
      gumbel_leaves_descend_kernel<decltype(g), false><<<blocks, SEL_WARPS * 32, 0, st>>>(*t, *gb, *b, d_issued, nullptr);
    return cuda_check(cudaGetLastError(), "gumbel_leaves_descend_kernel launch");
  });
  if (rc != FPC_OK) return rc;
  return observe_slots(t, b, batch_rotation, d_planes, flags, track, stream);
}

int fpc_tree_gumbel_result_leaves(const fpc_tree *t, const fpc_gumbel *gb, const int32_t *d_issued, int32_t *d_action,
                                  float *d_policy, void *stream) {
  int rc = check_tree(t, "fpc_tree_gumbel_result_leaves");
  if (rc == FPC_OK) rc = check_gumbel(t, gb, "fpc_tree_gumbel_result_leaves");
  if (rc != FPC_OK) return rc;
  if (t->n_games == 0) return FPC_OK;
  if (!d_issued || !d_action || !d_policy) return fail(FPC_ERR_ARG, "fpc_tree_gumbel_result_leaves: null issued / action / policy");
  const int blocks = (t->n_games + SEL_WARPS - 1) / SEL_WARPS;
  tree_gumbel_result_leaves_kernel<<<blocks, SEL_WARPS * 32, 0, (cudaStream_t)stream>>>(*t, *gb, d_issued, d_action, d_policy);
  return cuda_check(cudaGetLastError(), "tree_gumbel_result_leaves_kernel launch");
}

int fpc_tree_expand_backup_leaves(const fpc_tree *t, const fpc_leaf_batch *b, const float *d_logits,
                                  const float *d_values, void *stream) {
  int rc = check_tree(t, "fpc_tree_expand_backup_leaves");
  if (rc == FPC_OK) rc = check_batch(t, b, "fpc_tree_expand_backup_leaves");
  if (rc != FPC_OK) return rc;
  if (t->n_games == 0) return FPC_OK;
  if (!d_logits || !d_values) return fail(FPC_ERR_ARG, "fpc_tree_expand_backup_leaves: null logits / values");
  if (reinterpret_cast<uintptr_t>(d_logits) & 15) return fail(FPC_ERR_ARG, "logits must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  return dispatch(t->R, [&](auto g) {
    leaves_priors_kernel<decltype(g)><<<t->n_games * b->L, EXP_THREADS, 0, st>>>(*b, d_logits);
    CK(cudaGetLastError());
    leaves_commit_kernel<decltype(g)><<<t->n_games, LB_THREADS, 0, st>>>(*t, *b, d_values);
    return cuda_check(cudaGetLastError(), "leaves_commit_kernel launch");
  });
}

int fpc_tree_root_noise(const fpc_tree *t, uint64_t seed, const int64_t *d_keys, float alpha, float epsilon,
                        int32_t *d_done, void *stream) {
  int rc = check_tree(t, "fpc_tree_root_noise");
  if (rc != FPC_OK) return rc;
  if (!(alpha > 0.0f) || !std::isfinite(alpha))
    return fail(FPC_ERR_ARG, "fpc_tree_root_noise: alpha must be positive and finite, got " + std::to_string(alpha));
  if (!(epsilon >= 0.0f && epsilon <= 1.0f))
    return fail(FPC_ERR_ARG, "fpc_tree_root_noise: epsilon outside [0, 1]: " + std::to_string(epsilon));
  if (t->n_games == 0) return FPC_OK;
  if (!d_keys || !d_done) return fail(FPC_ERR_ARG, "fpc_tree_root_noise: null keys / done");
  const int blocks = (t->n_games + SEL_WARPS - 1) / SEL_WARPS;
  tree_root_noise_kernel<<<blocks, SEL_WARPS * 32, 0, (cudaStream_t)stream>>>(*t, seed, d_keys, (double)alpha,
                                                                              (double)epsilon, d_done);
  return cuda_check(cudaGetLastError(), "tree_root_noise_kernel launch");
}

int fpc_tree_sample_root(const fpc_tree *t, uint64_t seed, const int64_t *d_keys, double temperature, int32_t *d_action,
                         void *stream) {
  int rc = check_tree(t, "fpc_tree_sample_root");
  if (rc != FPC_OK) return rc;
  if (!(temperature > 0.0) || !std::isfinite(temperature))
    return fail(FPC_ERR_ARG, "fpc_tree_sample_root: temperature must be positive and finite, got " +
                                 std::to_string(temperature));
  if (!d_keys || !d_action) return fail(FPC_ERR_ARG, "fpc_tree_sample_root: null keys / action");
  if (t->n_games == 0) return FPC_OK;
  const int blocks = (t->n_games + SEL_WARPS - 1) / SEL_WARPS;
  tree_sample_root_kernel<<<blocks, SEL_WARPS * 32, 0, (cudaStream_t)stream>>>(*t, seed, d_keys, temperature, d_action);
  return cuda_check(cudaGetLastError(), "tree_sample_root_kernel launch");
}

}  // extern "C"
