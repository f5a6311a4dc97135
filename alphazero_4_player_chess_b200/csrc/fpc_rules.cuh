// The rules kernel body: one warp = one game (sm_100a; also compiled for the host by tests/host_emul, where a
// fibre-per-lane emulator runs this very code against the oracle).
//
// Legal moves are generated DIRECTLY -- no make / attack-test / undo per pseudo-legal move as in the reference
// (src/cpp/board.cpp:94-118 over engine/board.cpp:846-889) -- from three facts about the mover's king K:
//   * which enemy pieces attack K (the checkers),
//   * which of the mover's pieces are pinned to K by an enemy slider (they may only move along the pin line),
//   * which of K's eight neighbours are attacked once K has left its square.
// A non-king move is legal iff it keeps a pinned piece on its pin line and, when K is in check, captures the single
// checker or lands between it and K; a king step is legal iff its destination is not attacked; castling repeats
// the reference's own tests (engine/board.cpp:343-465 + the legal filter on the destination).  The result is the
// same SET of moves as the reference's filter (there is no en passant, so a move changes the attack picture of K only
// through its own from / to squares) -- pinned to the oracle on every playout, random and hand-made position of the
// test-suite -- at a fraction of the work: ~10 attack tests per position instead of one per pseudo-legal move.
//
// Board lookups use BIT line tables instead of byte rays: for each of the 64 lines of the 16x16 mailbox (16 rows,
// 16 columns, 16 diagonals, 16 anti-diagonals) one word holds the occupancy (pieces + walls) and the enemy pieces
// of the line, a second one the enemy sliders that move along it.  A ray is then one 4-byte shared-memory load
// and a find-first-set; the tables are built from the piece list with four atomicOr per piece.
#pragma once
#include "fpc_device.cuh"

namespace fpc {

struct ObserveParams {
  const uint8_t *boards_in;  // [n][REC]
  uint8_t *boards_out;       // playout: updated records (may alias boards_in)
  int n;
  int need_movegen;
  uint64_t *moves;      // [n][MAX_MOVES] or null
  int32_t *flat;        // [n][MAX_MOVES] or null
  int32_t *counts;      // [n] or null
  int32_t *status;      // [n] or null
  const int32_t *k;     // [n] or null
  int k_all;            // -1: own turn
  // The ones of the dense outputs of this call, one record per game and tensor: cells [n][CELL_STRIDE] u16 (the
  // cells of the input planes), flats [n][FLAT_STRIDE] u16 (the flat indices of the legal-move mask); null = tensor
  // not asked for.  expand_kernel turns the records into the dense f32 tensors (zero fill + ones).  With inc_planes /
  // inc_mask set the record is also read (in: what the tensor holds now) and the tensor is updated in place --
  // previous ones cleared, current ones set -- instead of being rewritten (FPC_FLAG_INCREMENTAL).
  uint16_t *cells, *flats;
  float *inc_planes, *inc_mask;
  // playout
  int playout;
  uint64_t seed;
  uint64_t *game;
  int32_t *ply;
  const uint8_t *start;
  int max_plies;
  uint64_t game_stride;
  uint64_t *chosen;
  unsigned long long *counters;
};

// Records of one game (u16 units, 16-byte aligned parts): [0] the number of entries, [8, ...) the entries --
// plane cell indices ch*R*R + row*R + col (already rotated; at most one per on-board square) or flat action indices
// (at most MAX_MOVES; the four promotions of a pawn move share one).
constexpr int CELL_FIRST = 8, CELL_MAX = 160, CELL_STRIDE = CELL_FIRST + CELL_MAX;      // 336 B
constexpr int FLAT_FIRST = 8, FLAT_STRIDE = FLAT_FIRST + ((MAX_MOVES + 7) / 8) * 8;    // 624 B
constexpr int STATUS_IN_CHECK = 0x100, STATUS_CAN_TAKE_KING = 0x200, STATUS_OVERFLOW = 0x400, STATUS_FINISHED = 0x800,
              STATUS_CHECK = 0x1000;

// ---- line geometry ------------------------------------------------------------------------------------------
// line 0 row (id R1, position C1; lo = W, hi = E), 1 column (id C1, position R1; lo = N, hi = S),
// 2 diagonal (id (R1-C1)&15, position C1; lo = NW, hi = SE), 3 anti-diagonal (id (R1+C1)&15, position C1; lo = SW, hi = NE).
// A diagonal id is shared by two real diagonals of the 16x16 torus, but the two parts are separated by border cells
// (always walls), so a scan from an on-board square never leaves its own part.
__host__ __device__ __forceinline__ int line_entry(int line, int m) {
  const int R1 = m >> 4, C1 = m & 15;
  const int id = line == 0 ? R1 : (line == 1 ? C1 : (line == 2 ? (R1 - C1) & 15 : (R1 + C1) & 15));
  return line * 16 + id;
}
__host__ __device__ __forceinline__ int line_pos(int line, int m) { return line == 1 ? m >> 4 : m & 15; }
// mailbox square of position `pos` on line entry `e`
__host__ __device__ __forceinline__ int line_square(int e, int pos) {
  const int line = e >> 4, id = e & 15;
  const int R1 = line == 0 ? id : (line == 1 ? pos : (line == 2 ? (id + pos) & 15 : (id - pos) & 15));
  const int C1 = line == 1 ? id : pos;
  return (R1 << 4) | C1;
}
// line of a queen direction (plane order N NW W SW S SE E NE): N/S column, W/E row, NW/SE diagonal, SW/NE anti-diagonal
__host__ __device__ __forceinline__ int line_of_dir(int dir) { return (0x3021 >> ((dir & 3) * 4)) & 3; }  // N->1 NW->2 W->0 SW->3

template <class G>
struct WallTab {
  uint32_t w[64];
  constexpr WallTab() : w{} {
    for (int e = 0; e < 64; ++e) {
      uint32_t m = 0;
      for (int pos = 0; pos < 16; ++pos) {
        const int line = e >> 4, id = e & 15;
        const int R1 = line == 0 ? id : (line == 1 ? pos : (line == 2 ? (id + pos) & 15 : (id - pos) & 15));
        const int C1 = line == 1 ? id : pos;
        if (!G::legal(R1 - 1, C1 - 1)) m |= 1u << pos;
      }
      w[e] = m;
    }
  }
};
template <class G>
__device__ const WallTab<G> kWalls = WallTab<G>();

// Per-warp shared-memory scratch (3.9 KB).
template <class G>
struct alignas(16) RulesScratch {
  uint32_t moves[MAX_MOVES + 4];  // compact moves (see pack_compact); aliased by the all-piece list before generation
  uint32_t tabA[64];              // per line: bits 0-15 occupancy (pieces + walls), bits 16-31 enemy pieces
  uint32_t tabB[64];              // per line: bits 0-15 enemy sliders moving along this line
  uint8_t mb[256];                // byte mailbox (rows), WALL outside the board
  uint8_t rec[256];               // raw record staging (in and out)
  uint16_t plist[160];            // the mover's pieces: mailbox square | piece byte << 8
  uint16_t cells[CELL_STRIDE];    // the ones this call leaves in the planes tensor
  uint16_t flats[FLAT_STRIDE];    // ... and in the mask tensor
  uint32_t pinbits[8];            // mailbox bit set: the mover's pieces pinned to its king
  uint32_t tbits[8];              // mailbox bit set: squares that answer a single check (the checker + the squares between)
  uint8_t rights[4];
  uint8_t king[4];                // mailbox square per colour, NO_SQ = captured
  int turn;
  int pad[3];
};

// Nearest occupied positions either side of position k on a line (walls guarantee both).
__device__ __forceinline__ void nearest(uint32_t occ, int k, int &pl, int &ph) {
  ph = fpc_ffs(occ & (0xfffeu << k)) - 1;
  pl = 31 - fpc_clz(occ & ((1u << k) - 1u));
}

// Enemy non-sliders around a square.  Neighbour slots: 0-7 the knight squares (engine/board.cpp:676-694, all eight
// whatever invalid_area is), 8-15 the adjacent squares in plane-order direction nb-8 (kings :753-772; pawns :697-750:
// RED attacks from SW / SE of the target, YELLOW from NW / NE, BLUE from NW / SW, GREEN from NE / SE).  A quarter is
// four slots; their mailbox deltas travel as four signed bytes.  A knight jump from an edge square may leave the
// mailbox (rows) or wrap into the wall column of the neighbouring row (columns): both read as WALL.
__device__ __forceinline__ uint32_t quarter_deltas(int sub) {
  // knights (dcol,drow) (-2,-1)(-2,1)(-1,-2)(-1,2) | (1,-2)(1,2)(2,-1)(2,1); adjacent N NW W SW | S SE E NE
  return sub == 0 ? 0x1FDF0EEEu : (sub == 1 ? 0x12F221E1u : (sub == 2 ? 0x0FFFEFF0u : 0xF1011110u));
}
__device__ __forceinline__ int quarter_square(int t, uint32_t deltas, int j) { return t + (int)(int8_t)(deltas >> (8 * j)); }
__device__ __forceinline__ bool neighbour_hit(uint32_t p, int sub, int j, int enemy_team) {
  const uint32_t m = p & 0xBCu, side = 0x80u | ((uint32_t)enemy_team << 5);  // presence, team and type bits
  if (sub < 2) return m == (side | (KNIGHT << 2));
  return m == (side | (KING << 2)) || (m == side && ((0xA0820A28u >> (8 * color_of(p) + (sub - 2) * 4 + j)) & 1u));
}

// One quarter of "is square t attacked by the enemy team" (engine/board.cpp:606-787 GetAttackers2, limit 1): the
// sliders on line `sub` through t plus neighbour slots 4*sub .. 4*sub+3.  The occupancy of line `pline` is patched
// (cleared pclr, set pset: position bit masks) to test a position after a king step or castling.
template <class G>
__device__ __forceinline__ bool attack_quarter(const RulesScratch<G> &s, int t, int sub, int enemy_team, int pline,
                                               uint32_t pclr, uint32_t pset) {
  const int e = line_entry(sub, t), k = line_pos(sub, t);
  uint32_t occ = s.tabA[e] & 0xffffu;
  const uint32_t es = s.tabB[e];
  const uint32_t deltas = quarter_deltas(sub);
  uint32_t nbp[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int sq = quarter_square(t, deltas, j);
    nbp[j] = (unsigned)sq < 256u ? s.mb[sq] : WALL;
  }
  if (sub == pline) occ = (occ & ~pclr) | pset;
  int pl, ph;
  nearest(occ, k, pl, ph);
  bool hit = ((es >> ph) | (es >> pl)) & 1u;
#pragma unroll
  for (int j = 0; j < 4; ++j) hit |= neighbour_hit(nbp[j], sub, j, enemy_team);
  return hit;
}

// A run of moves of one piece: to = from + delta * (first + 1 + j), plane = plane0 + first + j, j < cnt; or, with
// promo set (cnt = 4), the four promotions N, B, R, Q of the single move (first = 0) (engine/board.cpp:82-88).
struct Run2 {
  int delta, plane0, first, cnt, promo;
};

// Keep the moves of a run that land on a square of `bits` (the answer to a single check): at most one.
__device__ __forceinline__ void restrict_run(const uint32_t *bits, int from, Run2 &r) {
  if (r.cnt == 0) return;
  const int n = r.promo ? 1 : r.cnt;
  int found = -1;
  for (int j = 0; j < n && found < 0; ++j) {
    const int to = from + r.delta * (r.first + 1 + j);
    if ((bits[to >> 5] >> (to & 31)) & 1u) found = j;
  }
  if (found < 0) {
    r.cnt = 0;
  } else if (!r.promo) {
    r.first += found;
    r.cnt = 1;
  }
}

// Moves of the mover's piece (square `from`, piece byte p) along line `line`: two runs (lo / hi side).
// Sliders (engine/board.cpp:209-311), king steps (:313-341; `ksafe` bit 4*d = neighbour in direction d is a legal
// destination), pawns (:47-177: push and double push along the forward line, captures on the two forward diagonals,
// promotion on the colour's promotion line, no en passant), knights (:179-207: lines 0-3 carry jumps 2*line and
// 2*line+1; |drow| < invalid_area only).
template <class G>
__device__ __forceinline__ void gen_runs(const RulesScratch<G> &s, int from, uint32_t p, int line, uint32_t ksafe,
                                         Run2 &lo, Run2 &hi) {
  constexpr int R = G::R;
  const int type = type_of(p), color = color_of(p), team = team_of(p);
  const int R1 = from >> 4, C1 = from & 15;
  lo = Run2{0, 0, 0, 0, 0};
  hi = Run2{0, 0, 0, 0, 0};
  if (type == KNIGHT) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int k = 2 * line + h;
      const int dr = kdrow(k), dc = kdcol(k);
      Run2 &out = h ? hi : lo;
      if ((dr < 0 ? -dr : dr) >= G::IA) continue;
      const int tr = R1 + dr, tc = C1 + dc;
      if ((unsigned)tr > 15u || (unsigned)tc > 15u) continue;
      const uint32_t o = s.mb[(tr << 4) | tc];
      if (o == WALL || (present(o) && team_of(o) == team)) continue;
      out.delta = dr * 16 + dc;
      out.plane0 = 8 * (R - 1) + k;
      out.cnt = 1;
    }
    return;
  }
  // how far each side may move without / with a capture
  int move_lo = 0, move_hi = 0, cap_lo = 0, cap_hi = 0;
  const int dlo = (0x3102 >> (line * 4)) & 15, dhi = dlo + 4;  // plane-order direction of the lo side: W N NW SW
  bool pawn = false;
  if (type == PAWN) {
    pawn = true;
    // forward: RED N (column, lo) BLUE E (row, hi) YELLOW S (column, hi) GREEN W (row, lo)
    const int fline = color & 1 ? 0 : 1;
    const bool fwd_hi = color == 1 || color == 2;
    if (line == fline) {
      const bool home = color == 0 ? R1 == R - 1 : (color == 1 ? C1 == 2 : (color == 2 ? R1 == 2 : C1 == R - 1));
      (fwd_hi ? move_hi : move_lo) = home ? 2 : 1;
    } else if (line >= 2) {
      // captures: RED NW (dia lo), NE (anti hi); BLUE NE (anti hi), SE (dia hi); YELLOW SW (anti lo), SE (dia hi);
      // GREEN NW (dia lo), SW (anti lo)
      const bool side_hi = line == 2 ? (color == 1 || color == 2) : (color == 0 || color == 1);
      (side_hi ? cap_hi : cap_lo) = 1;
    }
  } else if (type == KING) {
    move_lo = cap_lo = (ksafe >> (4 * dlo)) & 1u;
    move_hi = cap_hi = (ksafe >> (4 * dhi)) & 1u;
  } else {
    const bool straight = line < 2;
    const bool ok = type == QUEEN || (type == ROOK ? straight : (type == BISHOP && !straight));
    move_lo = move_hi = cap_lo = cap_hi = ok ? 16 : 0;
  }
  if ((move_lo | move_hi | cap_lo | cap_hi) == 0) return;
  const int e = line_entry(line, from), k = line_pos(line, from);
  const uint32_t a = s.tabA[e];
  int pl, ph;
  nearest(a & 0xffffu, k, pl, ph);
  const int emp_lo = k - pl - 1, emp_hi = ph - k - 1;
  const int en_lo = (a >> (16 + pl)) & 1u, en_hi = (a >> (16 + ph)) & 1u;
  lo.cnt = (emp_lo < move_lo ? emp_lo : move_lo) + (en_lo && emp_lo < cap_lo);
  hi.cnt = (emp_hi < move_hi ? emp_hi : move_hi) + (en_hi && emp_hi < cap_hi);
  lo.delta = qdelta(dlo), hi.delta = qdelta(dhi);
  lo.plane0 = dlo * (R - 1), hi.plane0 = dhi * (R - 1);
  if (pawn) {
    // promotion line (:58-76): RED row R/4, YELLOW row 3R/4, BLUE col 3R/4, GREEN col R/4 (0-based); only single steps reach it
    Run2 &r = lo.cnt ? lo : hi;
    if (r.cnt == 1) {
      const int to = from + r.delta;
      const int tr = (to >> 4) - 1, tc = (to & 15) - 1;
      const bool promo = color == 0 ? tr == R / 4 : (color == 2 ? tr == 3 * R / 4 : (color == 1 ? tc == 3 * R / 4 : tc == R / 4));
      if (promo) r.promo = 1, r.cnt = 4;
    }
  }
}

// Castling candidate (engine/board.cpp:343-465), side 0 queenside / 1 kingside: the right, the rook (own team: the
// partner's counts, :437) on its square, the squares between empty.  Returns the unit step king -> rook as a plane
// direction, or -1.  The three attack tests (king square, crossed square, destination after the move) follow.
template <class G>
__device__ __forceinline__ int castle_candidate(const RulesScratch<G> &s, int from, int color, uint32_t rights, int side) {
  constexpr int R = G::R;
  const bool allowed = side ? (rights >> 6) & 1 : (rights >> 5) & 1;
  if (!allowed) return -1;
  // RED ks E(6)/qs W(2), BLUE ks S(4)/qs N(0), YELLOW ks W/qs E, GREEN ks N/qs S
  const int udir = color == 0 ? (side ? 6 : 2) : (color == 1 ? (side ? 4 : 0) : (color == 2 ? (side ? 2 : 6) : (side ? 0 : 4)));
  const int u = qdelta(udir);
  const int nb = side ? 2 : 3;
  const int r = (from >> 4) - 1, c = (from & 15) - 1;
  const int ur = (u + 24) / 16 - 1, uc = u - ur * 16;
  const int rr = r + ur * (nb + 1), rc = c + uc * (nb + 1);
  if ((unsigned)rr >= (unsigned)R || (unsigned)rc >= (unsigned)R) return -1;  // Relative() -> missing (engine/board.h:194-199)
  const uint32_t rook = s.mb[from + u * (nb + 1)];
  if (!present(rook) || type_of(rook) != ROOK || team_of(rook) != (color & 1)) return -1;
  for (int k = 1; k <= nb; ++k)
    if (s.mb[from + u * k] != EMPTY) return -1;
  return udir;
}

// chess::Board::MakeMove (engine/board.cpp:1028-1096) on the byte mailbox, for a generator move.
template <class G>
__device__ __forceinline__ void make_compact2(RulesScratch<G> &s, uint32_t mv) {
  int from, to, plane, promo, castle;
  unpack_compact<G>(mv, from, to, plane, promo, castle);
  const int turn = s.turn;
  const uint32_t piece = s.mb[from], cap = s.mb[to];
  const int type = type_of(piece);
  if (type == KING) {
    s.rights[turn] = 0x80;
  } else if ((type == ROOK || type == QUEEN) && plane < 8 * (G::R - 1) && !((plane / (G::R - 1)) & 1)) {
    const int ct = rook_location_type<G>(turn, G::sq_of_mb(from));
    const uint32_t cur = s.rights[turn];
    if (ct == 0 && ((cur >> 6) & 1)) s.rights[turn] = 0x80 | (cur & 0x20);
    else if (ct == 1 && ((cur >> 5) & 1)) s.rights[turn] = 0x80 | (cur & 0x40);
  }
  if (present(cap) && type_of(cap) == KING) s.king[color_of(cap)] = NO_SQ;
  s.mb[from] = (uint8_t)EMPTY;
  s.mb[to] = (uint8_t)(promo != NO_PIECE ? mk_piece(turn, promo) : piece);
  if (type == KING) s.king[turn] = (uint8_t)to;
  if (castle) {
    int rf, rt;
    castle_rook(from, to, castle, rf, rt);
    const uint32_t rook = s.mb[rf];
    s.mb[rf] = (uint8_t)EMPTY;
    s.mb[rt] = (uint8_t)rook;
  }
  s.turn = (turn + 1) & 3;
}

// ---- the warp ------------------------------------------------------------------------------------------------
template <class G>
__device__ void rules_warp(const ObserveParams &P, RulesScratch<G> &s, const int g, const int lane) {
  constexpr int R = G::R;
  const unsigned lt_mask = (1u << lane) - 1u;
  // playout bookkeeping is read up front: with zero-copy host buffers each load is a PCIe round trip
  const uint64_t game_id = P.playout ? P.game[g] : 0;
  const int ply = P.playout ? P.ply[g] : 0;

  // ---- stage the record; line tables <- walls -------------------------------------------------------------------
  if (lane < G::REC / 16)
    reinterpret_cast<uint4 *>(s.rec)[lane] = reinterpret_cast<const uint4 *>(P.boards_in + (size_t)g * G::REC)[lane];
  s.tabA[lane] = kWalls<G>.w[lane];
  s.tabA[lane + 32] = kWalls<G>.w[lane + 32];
  s.tabB[lane] = 0;
  s.tabB[lane + 32] = 0;
  if (lane < 8) s.pinbits[lane] = 0, s.tbits[lane] = 0;
  if (lane < 4) s.king[lane] = NO_SQ;
  __syncwarp();
  const int turn = s.rec[G::OFF_TURN] & 3;
  const int my_team = turn & 1, enemy_team = my_team ^ 1;
  if (lane < 4) s.rights[lane] = s.rec[G::OFF_RIGHTS + lane];
  if (lane == 0) s.turn = turn;

  // ---- scan: lane l owns mailbox cells 8l .. 8l+7 (row l/2, columns 8(l&1) ..): byte mailbox + the list of all pieces ----
  uint16_t *alist = reinterpret_cast<uint16_t *>(s.moves);
  int na = 0;
  {
    const int R1 = lane >> 1, r = R1 - 1;
    uint32_t b[8];
    uint32_t pres = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = (lane & 1) * 8 + j - 1;
      uint32_t p = WALL;
      if (G::legal(r, c)) {
        p = s.rec[r * R + c] & 0xFCu;
        if (!present(p)) p = EMPTY;  // one canonical empty byte
      }
      b[j] = p;
      pres |= (p >> 7) << j;
    }
    reinterpret_cast<uint2 *>(s.mb)[lane] =
        make_uint2(b[0] | (b[1] << 8) | (b[2] << 16) | (b[3] << 24), b[4] | (b[5] << 8) | (b[6] << 16) | (b[7] << 24));
    // exclusive prefix sum of the per-lane piece counts (<= 8), bit-sliced over four ballots
    const int mine = __popc(pres);
    int excl = 0;
#pragma unroll
    for (int bit = 0; bit < 4; ++bit) {
      const unsigned v = __ballot_sync(FULL, (mine >> bit) & 1);
      excl += __popc(v & lt_mask) << bit;
      na += __popc(v) << bit;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if ((pres >> j) & 1u) alist[excl++] = (uint16_t)((lane * 8 + j) | (b[j] << 8));
  }
  __syncwarp();

  // ---- every piece: line tables, king squares, the mover's piece list, the input-plane cells ----------------------
  const bool want_planes = P.cells != nullptr;
  int rot = 0;
  if (want_planes) {
    rot = P.k ? P.k[g] : (P.k_all < 0 ? turn : P.k_all);
    rot &= 3;
  }
  int np = 0;
  for (int base = 0; base < na; base += 32) {
    const int i = base + lane;
    const bool active = i < na;
    uint32_t e = 0;
    bool own = false;
    if (active) {
      e = alist[i];
      const int m = e & 0xff;
      const uint32_t p = e >> 8;
      const int type = type_of(p), color = color_of(p);
      const int R1 = m >> 4, C1 = m & 15;
      const bool enemy = team_of(p) != my_team;
      own = color == turn;
      const int e0 = R1, e1 = 16 + C1, e2 = 32 + ((R1 - C1) & 15), e3 = 48 + ((R1 + C1) & 15);
      const uint32_t va = enemy ? 0x10001u : 1u;
      atomicOr(&s.tabA[e0], va << C1);
      atomicOr(&s.tabA[e1], va << R1);
      atomicOr(&s.tabA[e2], va << C1);
      atomicOr(&s.tabA[e3], va << C1);
      if (enemy && (type == ROOK || type == QUEEN)) {
        atomicOr(&s.tabB[e0], 1u << C1);
        atomicOr(&s.tabB[e1], 1u << R1);
      }
      if (enemy && (type == BISHOP || type == QUEEN)) {
        atomicOr(&s.tabB[e2], 1u << C1);
        atomicOr(&s.tabB[e3], 1u << C1);
      }
      if (type == KING) s.king[color] = (uint8_t)m;
      if (want_planes) {
        // ch = ((color - turn) mod 4)*6 + type - 1, -1 wrapping to 23 (src/cpp/board.cpp:336)
        int ch = ((color - turn) & 3) * 6 + type - 1;
        if (ch < 0) ch += 24;
        // torch.rot90(k) on the last two dims: one quarter turn sends (r,c) -> (R-1-c, r)
        const int r = R1 - 1, c = C1 - 1;
        const int rr = rot == 0 ? r : (rot == 1 ? R - 1 - c : (rot == 2 ? R - 1 - r : c));
        const int cc = rot == 0 ? c : (rot == 1 ? r : (rot == 2 ? R - 1 - c : R - 1 - r));
        const int bit = ch * G::NSQ + rr * R + cc;
        if (i < CELL_MAX) s.cells[CELL_FIRST + i] = (uint16_t)bit;
      }
    }
    const unsigned ob = __ballot_sync(FULL, own);
    if (own) s.plist[np + __popc(ob & lt_mask)] = (uint16_t)e;
    np += __popc(ob);
  }
  const int n_cells = na;
  __syncwarp();

  int n_legal = 0, status = 0;
  uint32_t chosen_mv = 0;
  if (P.need_movegen) {
    const int king_sq = s.king[turn];
    int n_moves = 0, n_chk = 0;
    bool overflow = false, takes_king = false;
    const int ek1 = s.king[(turn + 1) & 3], ek2 = s.king[(turn + 3) & 3];
    if (king_sq != NO_SQ) {  // engine/board.cpp:852-856: no moves without a king
      // ---- the king: checkers, pins (lanes 0-3: one line each + four neighbour slots) ---------------------------
      {
        int chk = 0;
        if (lane < 4) {
          const int e = line_entry(lane, king_sq), k = line_pos(lane, king_sq);
          const uint32_t occ = s.tabA[e] & 0xffffu, es = s.tabB[e];
          int pl, ph;
          nearest(occ, k, pl, ph);
          const int dlo = (0x3102 >> (lane * 4)) & 15;
#pragma unroll
          for (int side = 0; side < 2; ++side) {
            const int p1 = side ? ph : pl;
            if ((es >> p1) & 1u) {
              // a slider gives check: it and the squares between answer the check
              ++chk;
              const int d = qdelta(side ? dlo + 4 : dlo), dist = side ? ph - k : k - pl;
              for (int j = 1; j <= dist; ++j) {
                const int sq = king_sq + d * j;
                atomicOr(&s.tbits[sq >> 5], 1u << (sq & 31));
              }
            } else {
              // pinned: the first piece is the mover's and the next one beyond it an enemy slider of this line
              const uint32_t beyond = side ? occ & (0xfffeu << p1) : occ & ((1u << p1) - 1u);
              if (beyond) {
                const int p2 = side ? fpc_ffs(beyond) - 1 : 31 - fpc_clz(beyond);
                if ((es >> p2) & 1u) {
                  const int sq = line_square(e, p1);
                  const uint32_t pc = s.mb[sq];
                  if (present(pc) && color_of(pc) == turn) atomicOr(&s.pinbits[sq >> 5], 1u << (sq & 31));
                }
              }
            }
          }
          const uint32_t deltas = quarter_deltas(lane);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int sq = quarter_square(king_sq, deltas, j);
            if ((unsigned)sq < 256u && neighbour_hit(s.mb[sq], lane, j, enemy_team)) {
              ++chk;
              atomicOr(&s.tbits[sq >> 5], 1u << (sq & 31));
            }
          }
        }
#pragma unroll
        for (int bit = 0; bit < 3; ++bit) n_chk += __popc(__ballot_sync(FULL, (chk >> bit) & 1)) << bit;
      }
      // ---- the king's eight neighbours: a legal destination is on the board, not the mover's team's, and not attacked
      //      once the king has left (lane = destination direction * 4 + quarter of the attack test) ----------------
      uint32_t ksafe = 0;
      {
        const int d = lane >> 2, sub = lane & 3;
        const int t = king_sq + qdelta(d);
        const uint32_t cellv = s.mb[t];
        const bool cand = cellv != WALL && !(present(cellv) && team_of(cellv) == my_team);
        bool hit = false;
        if (cand) {
          const int kl = line_of_dir(d);
          hit = attack_quarter<G>(s, t, sub, enemy_team, kl, 1u << line_pos(kl, king_sq), 0u);
        }
        const unsigned hb = __ballot_sync(FULL, hit), cb = __ballot_sync(FULL, cand);
        ksafe = cb & ~(hb | (hb >> 1) | (hb >> 2) | (hb >> 3)) & 0x11111111u;  // bit 4*d: direction d is a legal king step
      }
      __syncwarp();  // pinbits / tbits complete

      // ---- generation: lane = (piece, line), two runs of moves each; written out with a warp prefix sum -----------
      if (n_chk >= 2) {  // double check: only the king moves
        if (lane == 0) s.plist[0] = (uint16_t)(king_sq | (s.mb[king_sq] << 8));
        np = 1;
        __syncwarp();
      }
      const int items = np * 4;
      constexpr uint32_t KEY_STEP = (uint32_t)(G::NSQ * 8) << 14;  // one plane further in the compact move
      for (int base = 0; base < items; base += 32) {
        const int item = base + lane;
        Run2 lo{0, 0, 0, 0, 0}, hi{0, 0, 0, 0, 0};
        int from = 0;
        if (item < items) {
          const uint32_t e = s.plist[item >> 2];
          from = e & 0xff;
          const uint32_t p = e >> 8;
          const int line = item & 3;
          gen_runs<G>(s, from, p, line, ksafe, lo, hi);
          if (type_of(p) != KING) {
            if ((s.pinbits[from >> 5] >> (from & 31)) & 1u) {
              // pinned: only along the line it shares with the king (a knight has none)
              const int KR = king_sq >> 4, KC = king_sq & 15, R1 = from >> 4, C1 = from & 15;
              const int pin_line = R1 == KR ? 0 : (C1 == KC ? 1 : (R1 - C1 == KR - KC ? 2 : 3));
              if (type_of(p) == KNIGHT || line != pin_line) lo.cnt = hi.cnt = 0;
            }
            if (n_chk == 1) {
              restrict_run(s.tbits, from, lo);
              restrict_run(s.tbits, from, hi);
            }
          }
        }
        const int cnt = lo.cnt + hi.cnt;  // <= 26: two rays of at most 13 squares
        // a king capture counts whether or not this round fits the buffer (only the last square of a run can hold a piece)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const Run2 &r = h ? hi : lo;
          const int to0 = from + r.delta * (r.first + 1);
          const int last = r.promo ? to0 : to0 + r.delta * (r.cnt - 1);
          takes_king |= r.cnt > 0 && (last == ek1 || last == ek2);
        }
        int excl = 0, total = 0;
#pragma unroll
        for (int bit = 0; bit < 5; ++bit) {
          const unsigned v = __ballot_sync(FULL, (cnt >> bit) & 1);
          excl += __popc(v & lt_mask) << bit;
          total += __popc(v) << bit;
        }
        if (n_moves + total > MAX_MOVES) {
          overflow = true;
        } else {
          int at = n_moves + excl;
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const Run2 &r = h ? hi : lo;
            if (r.cnt == 0) continue;
            // the run's moves differ by a constant: one plane and one step further (promotions: the piece type)
            const int to0 = from + r.delta * (r.first + 1);
            uint32_t mv = pack_compact<G>(from, to0, r.plane0 + r.first, r.promo ? KNIGHT : NO_PIECE, 0);
            const uint32_t inc = r.promo ? 1u << 14 : KEY_STEP + (uint32_t)r.delta;
            for (int j = 0; j < r.cnt; ++j, mv += inc) s.moves[at++] = mv;
          }
          n_moves += total;
        }
      }
      // ---- castling (engine/board.cpp:343-465): never out of check; the crossed square and (after the move) the
      //      destination must not be attacked.  lane = side * 8 + which * 4 + quarter ------------------------------
      {
        int udir = -1;
        if (lane < 16 && n_chk == 0) udir = castle_candidate<G>(s, king_sq, turn, s.rights[turn], lane >> 3);
        if (__any_sync(FULL, udir >= 0)) {
          bool hit = false;
          if (udir >= 0) {
            const int side = lane >> 3, which = (lane >> 2) & 1, sub = lane & 3;
            const int u = qdelta(udir), kl = line_of_dir(udir);
            if (which == 0) {
              hit = attack_quarter<G>(s, king_sq + u, sub, enemy_team, -1, 0u, 0u);  // :456, on the board as it stands
            } else {
              // after the move: king on from+2u, rook on from+u, both origin squares empty
              const int rook_from = king_sq + u * (side ? 3 : 4);
              const uint32_t clr = (1u << line_pos(kl, king_sq)) | (1u << line_pos(kl, rook_from));
              hit = attack_quarter<G>(s, king_sq + 2 * u, sub, enemy_team, kl, clr, 1u << line_pos(kl, king_sq + u));
            }
          }
          const unsigned hb = __ballot_sync(FULL, hit);
          uint32_t mv = 0;
          if ((lane == 0 || lane == 8) && udir >= 0 && ((hb >> lane) & 0xffu) == 0)
            mv = pack_compact<G>(king_sq, king_sq + 2 * qdelta(udir), udir * (R - 1) + 1, NO_PIECE, lane ? 2 : 1);
          const unsigned cb = __ballot_sync(FULL, mv != 0);
          if (cb) {
            if (n_moves + __popc(cb) > MAX_MOVES) {
              overflow = true;
            } else {
              if (mv) s.moves[n_moves + __popc(cb & lt_mask)] = mv;
              n_moves += __popc(cb);
            }
          }
        }
      }
      __syncwarp();
    }
    n_legal = n_moves;
    takes_king = __any_sync(FULL, takes_king);

    // ---- result (engine/board.cpp:891-939, order-independent contract) ---------------------
    const bool ry = my_team == 0;
    int result = 0;
    if (king_sq == NO_SQ) {
      result = ry ? 2 : 1;
    } else if (n_legal == 0 && !overflow) {
      result = n_chk ? (ry ? 2 : 1) : 3;
      if (n_chk) status |= STATUS_IN_CHECK;
    }
    status |= result;
    if (n_chk) status |= STATUS_CHECK;
    if (takes_king) status |= STATUS_CAN_TAKE_KING;
    if (overflow) status |= STATUS_OVERFLOW;

    // ---- canonical order: rank = number of smaller keys (keys are unique) ------------------
    uint32_t pick = 0xffffffffu;
    if (P.playout && result == 0)
      pick = (uint32_t)(((mix64(P.seed, game_id, (uint64_t)ply) >> 32) * (uint64_t)n_legal) >> 32);
    const bool want_lists = P.moves || P.flat;
    const bool want_flats = P.flats != nullptr;
    if ((want_lists || P.playout || want_flats) && n_legal <= 32) {
      // one move per lane: a 15-step bitonic network over the warp leaves lane i with the i-th smallest key
      __syncwarp();
      uint32_t mv = lane < n_legal ? s.moves[lane] : 0xffffffffu;
      if (want_lists || P.playout) {
#pragma unroll
        for (int k = 2; k <= 32; k <<= 1)
#pragma unroll
          for (int j = k >> 1; j > 0; j >>= 1) {
            const uint32_t other = __shfl_xor_sync(FULL, mv, j);
            const bool keep_min = ((lane & j) == 0) == ((lane & k) == 0);
            mv = keep_min ? (mv < other ? mv : other) : (mv > other ? mv : other);
          }
      }
      if (lane < n_legal) {
        const uint32_t flat = mv >> 17;
        if (want_flats) s.flats[FLAT_FIRST + lane] = (uint16_t)flat;
        if (P.moves) P.moves[(size_t)g * MAX_MOVES + lane] = expand_move<G>(s.mb, s.rights, mv);
        if (P.flat) P.flat[(size_t)g * MAX_MOVES + lane] = (int32_t)flat;
        if ((uint32_t)lane == pick) chosen_mv = mv;
      }
      __syncwarp();
    } else if (want_lists || P.playout || want_flats) {
      // pad to a multiple of four with keys above every real one: the rank loop compares four keys per load
      if (lane < 4) s.moves[n_legal + lane] = 0xffffffffu;
      __syncwarp();
      for (int base = 0; base < n_legal; base += 32) {
        const int i = base + lane;
        if (i < n_legal) {
          const uint32_t mv = s.moves[i];
          const uint32_t flat = mv >> 17;
          if (want_flats) s.flats[FLAT_FIRST + i] = (uint16_t)flat;
          if (want_lists || P.playout) {
            int rank = 0;
            for (int j = 0; j < n_legal; j += 4) {
              const uint4 q = *reinterpret_cast<const uint4 *>(&s.moves[j]);
              rank += (q.x < mv) + (q.y < mv) + (q.z < mv) + (q.w < mv);
            }
            if (P.moves) P.moves[(size_t)g * MAX_MOVES + rank] = expand_move<G>(s.mb, s.rights, mv);
            if (P.flat) P.flat[(size_t)g * MAX_MOVES + rank] = (int32_t)flat;
            if ((uint32_t)rank == pick) chosen_mv = mv;
          }
        }
      }
      __syncwarp();
    }
    if (lane == 0) {
      if (P.counts) P.counts[g] = n_legal;
    }
  }

  // ---- the records of ones / in-place update of the dense tensors (FPC_FLAG_INCREMENTAL) ---------
  if (P.cells || P.flats) {
    uint16_t *gc = P.cells ? P.cells + (size_t)g * CELL_STRIDE : nullptr;
    uint16_t *gf = P.flats ? P.flats + (size_t)g * FLAT_STRIDE : nullptr;
    const int new_cells = n_cells > CELL_MAX ? CELL_MAX : n_cells, new_flats = n_legal;
    if (P.inc_planes && gc) {
      float *dst = P.inc_planes + (size_t)g * G::SSZ;
      const int old = gc[0];
      for (int i = lane; i < old; i += 32) dst[gc[CELL_FIRST + i]] = 0.0f;
    }
    if (P.inc_mask && gf) {
      float *dst = P.inc_mask + (size_t)g * G::ASZ;
      const int old = gf[0];
      for (int i = lane; i < old; i += 32) dst[gf[FLAT_FIRST + i]] = 0.0f;
    }
    if (lane == 0) s.cells[0] = (uint16_t)new_cells, s.flats[0] = (uint16_t)new_flats;
    __syncwarp();  // warp-level memory ordering: every clear precedes every set (a cell may be in both records)
    if (P.inc_planes && gc) {
      float *dst = P.inc_planes + (size_t)g * G::SSZ;
      for (int i = lane; i < new_cells; i += 32) dst[s.cells[CELL_FIRST + i]] = 1.0f;
    }
    if (P.inc_mask && gf) {
      float *dst = P.inc_mask + (size_t)g * G::ASZ;
      for (int i = lane; i < new_flats; i += 32) dst[s.flats[FLAT_FIRST + i]] = 1.0f;
    }
    // only the used part of a record travels
    if (gc)
      for (int i = lane; i < (CELL_FIRST + new_cells + 7) / 8; i += 32) reinterpret_cast<uint4 *>(gc)[i] = reinterpret_cast<const uint4 *>(s.cells)[i];
    if (gf)
      for (int i = lane; i < (FLAT_FIRST + new_flats + 7) / 8; i += 32) reinterpret_cast<uint4 *>(gf)[i] = reinterpret_cast<const uint4 *>(s.flats)[i];
  }

  // ---- playout: play the chosen move or re-seed the slot ------------------------------------
  if (P.playout) {
    const unsigned who = __ballot_sync(FULL, chosen_mv != 0);
    const int result = status & 3;
    uint64_t chosen64 = 0;
    bool finished = false;
    if (result == 0 && who) {
      const uint32_t mv = __shfl_sync(FULL, chosen_mv, __ffs(who) - 1);
      if (P.chosen) chosen64 = expand_move<G>(s.mb, s.rights, mv);
      __syncwarp();
      if (lane == 0) make_compact2<G>(s, mv);
      __syncwarp();
      if (ply + 1 >= P.max_plies) finished = true;
    } else {
      finished = true;
    }
    if (finished) {
      status |= STATUS_FINISHED;
      if (lane < G::REC / 16)
        reinterpret_cast<uint4 *>(P.boards_out + (size_t)g * G::REC)[lane] =
            __ldg(reinterpret_cast<const uint4 *>(P.start) + lane);
    } else {
      // mailbox -> record: lane l < 2R packs half a row
      if (lane < 2 * R) {
        const int row = lane >> 1, c0 = (lane & 1) * ((R + 1) / 2);
#pragma unroll
        for (int j = 0; j < (R + 1) / 2; ++j) {
          const int c = c0 + j;
          if (c < R) s.rec[row * R + c] = G::legal(row, c) ? s.mb[G::mb(row, c)] : (uint8_t)EMPTY;
        }
      }
      if (lane < G::REC - G::NSQ) {
        const int i = G::NSQ + lane;
        uint32_t v = 0;
        if (i == G::OFF_TURN) {
          v = s.turn;
        } else if (i < G::OFF_KING) {
          v = s.rights[i - G::OFF_RIGHTS];
        } else if (i < G::OFF_KING + 4) {
          const int k = s.king[i - G::OFF_KING];
          v = k == NO_SQ ? G::NSQ : G::sq_of_mb(k);
        }
        s.rec[i] = (uint8_t)v;
      }
      __syncwarp();
      if (lane < G::REC / 16)
        reinterpret_cast<uint4 *>(P.boards_out + (size_t)g * G::REC)[lane] = reinterpret_cast<const uint4 *>(s.rec)[lane];
    }
    if (lane == 0) {
      if (P.chosen) P.chosen[g] = chosen64;
      if (finished) {
        P.game[g] = game_id + P.game_stride;
        P.ply[g] = 0;
      } else {
        P.ply[g] = ply + 1;
      }
      if (P.counters) {
        atomicAdd(&P.counters[0], 1ull);
        atomicAdd(&P.counters[6], (unsigned long long)n_legal);
        if (finished) {
          atomicAdd(&P.counters[1], 1ull);
          atomicAdd(&P.counters[2 + result], 1ull);
        }
        if (status & STATUS_OVERFLOW) atomicAdd(&P.counters[7], 1ull);
      }
    }
  }
  if (lane == 0 && P.status) P.status[g] = status;
}

}  // namespace fpc
