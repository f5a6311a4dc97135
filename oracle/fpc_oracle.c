/* TEST INFRASTRUCTURE -- not product code.
 *
 * CPU restatement ("port") of the reference hot path of jorr3/Alphazero-4-player-chess in
 * plain C11, geometry (R = rows = cols, IA = invalid_area) passed at run time.  Every
 * function cites the reference file:line it follows (paths relative to /root/reference).
 *
 * PINNING: the reference ships no tests or golden vectors (SURVEY 4).  This restatement is
 * pinned against the reference ITSELF run in the build container: (1) the unmodified rules
 * engine compiled by oracle/Makefile into oracle/_ref/ (perft tables, legal-move sets, post-move
 * boards, results over random playouts at four geometries: tests/test_oracle_vs_ref.py), and
 * (2) fixtures dumped from the reference's own pybind module for the encoder, the mask and the
 * MCTS node statistics (tests/golden/, generator: tests/golden/make_golden.py).
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may load this library;
 * the product path never does.
 *
 * Board record: see include/fpc.h.  Moves are the reference's 8-byte chess::Move image
 * (src/cpp/engine/board.h:419-435), little-endian u64:
 *   byte0 from, byte1 to, byte2 captured Piece bits (0x18 = none), byte3 promotion type
 *   (6 = none), byte4/5 rook from/to (R*R = none), byte6 rights before, byte7 rights after
 *   (0 = absent, else 0x80 | ks<<6 | qs<<5).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

enum { PAWN = 0, KNIGHT = 1, BISHOP = 2, ROOK = 3, QUEEN = 4, KING = 5, NO_PIECE = 6 };
enum { RED = 0, BLUE = 1, YELLOW = 2, GREEN = 3 };
enum { IN_PROGRESS = 0, WIN_RY = 1, WIN_BG = 2, STALEMATE = 3 };
#define EMPTY 0x18
#define MAX_MOVES 300 /* engine/board.h:706 move_buffer_size_ */

typedef struct {
  int R, IA, nsq, rec, off_turn, off_rights, off_king;
} Geo;

static Geo geo(int R, int IA) {
  Geo g;
  g.R = R;
  g.IA = IA;
  g.nsq = R * R;
  g.rec = ((g.nsq + 12 + 15) / 16) * 16;
  g.off_turn = g.nsq;
  g.off_rights = g.nsq + 1;
  g.off_king = g.nsq + 5;
  return g;
}

/* engine/board.h:101-130 */
static inline int present(uint8_t p) { return (p & 0x80) != 0; }
static inline int color_of(uint8_t p) { return (p >> 5) & 3; }
static inline int type_of(uint8_t p) { return (p >> 2) & 7; }
static inline int team_of_color(int c) { return c & 1; } /* engine/board.h:64-67 */
static inline int team_of(uint8_t p) { return team_of_color(color_of(p)); }
static inline uint8_t mk_piece(int color, int type) { return (uint8_t)(0x80 | (color << 5) | (type << 2)); }
static inline uint8_t mk_rights(int ks, int qs) { return (uint8_t)(0x80 | (ks << 6) | (qs << 5)); }

/* engine/board.h:647-654 */
static int legal_loc(const Geo *g, int row, int col) {
  int maxr = g->R - 1, maxc = g->R - 1;
  if (row < 0 || row > maxr || col < 0 || col > maxc ||
      (row < g->IA && (col < g->IA || col > maxc - g->IA)) ||
      (row > maxr - g->IA && (col < g->IA || col > maxc - g->IA)))
    return 0;
  return 1;
}

static inline uint64_t pack_move(int from, int to, uint8_t cap, int promo, int rook_from, int rook_to,
                                 uint8_t r0, uint8_t r1) {
  return (uint64_t)(uint8_t)from | ((uint64_t)(uint8_t)to << 8) | ((uint64_t)cap << 16) |
         ((uint64_t)(uint8_t)promo << 24) | ((uint64_t)(uint8_t)rook_from << 32) |
         ((uint64_t)(uint8_t)rook_to << 40) | ((uint64_t)r0 << 48) | ((uint64_t)r1 << 56);
}
#define MV_FROM(m) ((int)((m) & 0xff))
#define MV_TO(m) ((int)(((m) >> 8) & 0xff))
#define MV_CAP(m) ((uint8_t)(((m) >> 16) & 0xff))
#define MV_PROMO(m) ((int)(((m) >> 24) & 0xff))
#define MV_RFROM(m) ((int)(((m) >> 32) & 0xff))
#define MV_RTO(m) ((int)(((m) >> 40) & 0xff))
#define MV_R0(m) ((uint8_t)(((m) >> 48) & 0xff))
#define MV_R1(m) ((uint8_t)(((m) >> 56) & 0xff))

typedef struct {
  uint64_t *buf;
  int n, cap;
} MoveList;

static void push(MoveList *ml, uint64_t m) {
  if (ml->n < ml->cap) ml->buf[ml->n] = m;
  ml->n++;
}

/* engine/board.cpp:47-93 AddPawnMoves2 (en-passant arguments are dropped by the Move ctor,
 * engine/board.h:349-359). */
static void add_pawn_moves(const Geo *g, MoveList *ml, int from, int to, int color, uint8_t cap) {
  int R = g->R, promo = 0;
  int trow = to / R, tcol = to % R;
  switch (color) {
    case RED: promo = trow == R / 4; break;
    case BLUE: promo = tcol == 3 * R / 4; break;
    case YELLOW: promo = trow == 3 * R / 4; break;
    case GREEN: promo = tcol == R / 4; break;
  }
  if (promo) {
    push(ml, pack_move(from, to, cap, KNIGHT, g->nsq, g->nsq, 0, 0));
    push(ml, pack_move(from, to, cap, BISHOP, g->nsq, g->nsq, 0, 0));
    push(ml, pack_move(from, to, cap, ROOK, g->nsq, g->nsq, 0, 0));
    push(ml, pack_move(from, to, cap, QUEEN, g->nsq, g->nsq, 0, 0));
  } else {
    push(ml, pack_move(from, to, cap, NO_PIECE, g->nsq, g->nsq, 0, 0));
  }
}

/* engine/board.cpp:97-177 GetPawnMoves2 */
static void pawn_moves(const Geo *g, const uint8_t *b, MoveList *ml, int from, uint8_t piece) {
  int R = g->R, color = color_of(piece), team = team_of(piece);
  int row = from / R, col = from % R, dr = 0, dc = 0, not_moved = 0;
  switch (color) {
    case RED: dr = -1; not_moved = row == R - 2; break;
    case BLUE: dc = 1; not_moved = col == 1; break;
    case YELLOW: dr = 1; not_moved = row == 1; break;
    case GREEN: dc = -1; not_moved = col == R - 2; break;
  }
  if (legal_loc(g, row + dr, col + dc)) {
    int to = (row + dr) * R + col + dc;
    if (!present(b[to])) {
      add_pawn_moves(g, ml, from, to, color, EMPTY);
      if (not_moved) {
        /* the reference reads the double-step square without a bounds check (:143-144);
         * it is always on the board when the single step was (home rank/file geometry). */
        int r2 = row + 2 * dr, c2 = col + 2 * dc;
        if (r2 >= 0 && r2 < R && c2 >= 0 && c2 < R) {
          int to2 = r2 * R + c2;
          if (!present(b[to2])) add_pawn_moves(g, ml, from, to2, color, EMPTY);
        }
      }
    }
  }
  int check_cols = team == 0;
  for (int incr = 0; incr < 2; ++incr) {
    int cr = row + dr, cc = col + dc;
    if (check_cols) cc += incr == 0 ? -1 : 1;
    else cr += incr == 0 ? -1 : 1;
    if (legal_loc(g, cr, cc)) {
      uint8_t other = b[cr * R + cc];
      if (present(other) && team_of(other) != team) add_pawn_moves(g, ml, from, cr * R + cc, color, other);
    }
  }
}

/* engine/board.cpp:179-207 GetKnightMoves2 -- abs_delta_row runs 1..IA-1 (:188), so only the
 * (+-1,+-2) jumps exist when IA == 2. */
static void knight_moves(const Geo *g, const uint8_t *b, MoveList *ml, int from, uint8_t piece) {
  int R = g->R, row = from / R, col = from % R;
  for (int prs = 0; prs < 2; ++prs)
    for (int adr = 1; adr < g->IA; ++adr) {
      int dr = prs > 0 ? adr : -adr;
      for (int pcs = 0; pcs < 2; ++pcs) {
        int adc = adr == 1 ? 2 : 1;
        int dc = pcs > 0 ? adc : -adc;
        if (legal_loc(g, row + dr, col + dc)) {
          int to = (row + dr) * R + col + dc;
          uint8_t cap = b[to];
          if (!present(cap) || team_of(cap) != team_of(piece))
            push(ml, pack_move(from, to, cap, NO_PIECE, g->nsq, g->nsq, 0, 0));
        }
      }
    }
}

/* engine/board.cpp:209-238 AddMovesFromIncrMovement2 */
static void ray_moves(const Geo *g, const uint8_t *b, MoveList *ml, uint8_t piece, int from, int ir, int ic,
                      uint8_t r0, uint8_t r1) {
  int R = g->R, row = from / R + ir, col = from % R + ic;
  while (legal_loc(g, row, col)) {
    int to = row * R + col;
    uint8_t cap = b[to];
    if (!present(cap)) {
      push(ml, pack_move(from, to, EMPTY, NO_PIECE, g->nsq, g->nsq, r0, r1));
    } else {
      if (team_of(cap) != team_of(piece)) push(ml, pack_move(from, to, cap, NO_PIECE, g->nsq, g->nsq, r0, r1));
      break;
    }
    row += ir;
    col += ic;
  }
}

/* engine/board.cpp:240-254 */
static void bishop_moves(const Geo *g, const uint8_t *b, MoveList *ml, int from, uint8_t piece) {
  for (int pr = 0; pr < 2; ++pr)
    for (int pc = 0; pc < 2; ++pc) ray_moves(g, b, ml, piece, from, pr ? 1 : -1, pc ? 1 : -1, 0, 0);
}

/* engine/board.cpp:23-30 initial rook squares; :1474-1524 GetRookLocationType.
 * returns 0 kingside, 1 queenside, -1 neither */
static int rook_location_type(const Geo *g, int color, int sq) {
  int R = g->R, IA = g->IA, ks, qs;
  switch (color) {
    case RED: ks = (R - 1) * R + (R - 4); qs = (R - 1) * R + IA; break;
    case BLUE: ks = (R - 4) * R + 0; qs = IA * R + 0; break;
    case YELLOW: ks = 0 * R + IA; qs = 0 * R + (R - 4); break;
    default: ks = IA * R + (R - 1); qs = (R - 4) * R + (R - 1); break;
  }
  if (sq == ks) return 0;
  if (sq == qs) return 1;
  return -1;
}

/* engine/board.cpp:256-302 GetRookMoves2 (also reached for queens through :304-311, so a queen
 * standing on its colour's rook home square carries the same rights update). */
static void rook_moves(const Geo *g, const uint8_t *b, MoveList *ml, int from, uint8_t piece) {
  uint8_t r0 = 0, r1 = 0;
  int ct = rook_location_type(g, color_of(piece), from);
  if (ct >= 0) {
    uint8_t cur = b[g->off_rights + color_of(piece)];
    int ks = (cur >> 6) & 1, qs = (cur >> 5) & 1;
    if (ks || qs) {
      if (ct == 0) {
        if (ks) { r0 = cur; r1 = mk_rights(0, qs); }
      } else {
        if (qs) { r0 = cur; r1 = mk_rights(ks, 0); }
      }
    }
  }
  for (int dp = 0; dp < 2; ++dp) {
    int incr = dp > 0 ? 1 : -1;
    for (int dir = 0; dir < 2; ++dir) {
      int ir = dir > 0 ? incr : 0, ic = dir > 0 ? 0 : incr;
      ray_moves(g, b, ml, piece, from, ir, ic, r0, r1);
    }
  }
}

/* engine/board.cpp:606-777 GetAttackers2 with limit 1 == IsAttackedByTeam (:779-787) */
static int attacked_by_team(const Geo *g, const uint8_t *b, int team, int sq) {
  int R = g->R, lr = sq / R, lc = sq % R;
  /* rooks & queens: bounded by the R x R box only (:632) */
  for (int dir = 0; dir < 2; ++dir)
    for (int pos = 0; pos < 2; ++pos) {
      int ri = dir ? (pos ? 1 : -1) : 0, ci = dir ? 0 : (pos ? 1 : -1);
      int r = lr + ri, c = lc + ci;
      while (r >= 0 && r < R && c >= 0 && c < R) {
        uint8_t p = b[r * R + c];
        if (present(p)) {
          if (team_of(p) == team && (type_of(p) == ROOK || type_of(p) == QUEEN)) return 1;
          break;
        }
        r += ri;
        c += ci;
      }
    }
  /* bishops & queens: bounded by IsLegalLocation (:658) */
  for (int pr = 0; pr < 2; ++pr)
    for (int pc = 0; pc < 2; ++pc) {
      int ri = pr ? 1 : -1, ci = pc ? 1 : -1, r = lr + ri, c = lc + ci;
      while (legal_loc(g, r, c)) {
        uint8_t p = b[r * R + c];
        if (present(p)) {
          if (team_of(p) == team && (type_of(p) == BISHOP || type_of(p) == QUEEN)) return 1;
          break;
        }
        r += ri;
        c += ci;
      }
    }
  /* knights: all eight, whatever IA is (:676-694) */
  for (int rl = 0; rl < 2; ++rl)
    for (int pr = 0; pr < 2; ++pr) {
      int r = lr + (rl ? (pr ? 1 : -1) : (pr ? 2 : -2));
      for (int pc = 0; pc < 2; ++pc) {
        int c = lc + (rl ? (pc ? 2 : -2) : (pc ? 1 : -1));
        if (legal_loc(g, r, c)) {
          uint8_t p = b[r * R + c];
          if (present(p) && team_of(p) == team && type_of(p) == KNIGHT) return 1;
        }
      }
    }
  /* pawns (:697-750) */
  for (int pr = 0; pr < 2; ++pr) {
    int r = pr ? lr + 1 : lr - 1;
    if (r < 0 || r >= R) continue;
    for (int pc = 0; pc < 2; ++pc) {
      int c = pc ? lc + 1 : lc - 1;
      if (c < 0 || c >= R) continue;
      uint8_t p = b[r * R + c];
      if (present(p) && team_of(p) == team && type_of(p) == PAWN) {
        int a = 0;
        switch (color_of(p)) {
          case RED: a = pr; break;
          case BLUE: a = !pc; break;
          case YELLOW: a = !pr; break;
          case GREEN: a = pc; break;
        }
        if (a) return 1;
      }
    }
  }
  /* kings (:753-772) */
  for (int dr = -1; dr < 2; ++dr)
    for (int dc = -1; dc < 2; ++dc) {
      if (!dr && !dc) continue;
      if (legal_loc(g, lr + dr, lc + dc)) {
        uint8_t p = b[(lr + dr) * R + lc + dc];
        if (present(p) && team_of(p) == team && type_of(p) == KING) return 1;
      }
    }
  return 0;
}

/* engine/board.cpp:313-466 GetKingMoves2 */
static void king_moves(const Geo *g, const uint8_t *b, MoveList *ml, int from, uint8_t piece) {
  int R = g->R, row = from / R, col = from % R, color = color_of(piece);
  uint8_t r0 = b[g->off_rights + color], r1 = mk_rights(0, 0);
  for (int dr = -1; dr < 2; ++dr)
    for (int dc = -1; dc < 2; ++dc) {
      if (!dr && !dc) continue;
      if (legal_loc(g, row + dr, col + dc)) {
        int to = (row + dr) * R + col + dc;
        uint8_t cap = b[to];
        if (!present(cap) || team_of(cap) != team_of(piece))
          push(ml, pack_move(from, to, cap, NO_PIECE, g->nsq, g->nsq, r0, r1));
      }
    }
  int other_team = 1 - team_of(piece);
  for (int is_ks = 0; is_ks < 2; ++is_ks) {
    int allowed = is_ks ? (r0 >> 6) & 1 : (r0 >> 5) & 1;
    if (!allowed) continue;
    /* unit step from the king towards the rook, per colour (:352-433) */
    int ur = 0, uc = 0;
    switch (color) {
      case RED: uc = is_ks ? 1 : -1; break;
      case BLUE: ur = is_ks ? 1 : -1; break;
      case YELLOW: uc = is_ks ? -1 : 1; break;
      case GREEN: ur = is_ks ? -1 : 1; break;
    }
    int nb = is_ks ? 2 : 3; /* squares between */
    int rr = row + ur * (nb + 1), rc = col + uc * (nb + 1);
    /* BoardLocation::Relative yields "missing" off the box (engine/board.h:194-199); the
     * reference then reads one byte past the square array, which is never a rook. */
    if (rr < 0 || rr >= R || rc < 0 || rc >= R) continue;
    uint8_t rook = b[rr * R + rc];
    if (!present(rook) || type_of(rook) != ROOK || team_of(rook) != team_of(piece)) continue;
    int between = 0;
    for (int k = 1; k <= nb; ++k)
      if (present(b[(row + ur * k) * R + col + uc * k])) { between = 1; break; }
    if (between) continue;
    int sq1 = (row + ur) * R + col + uc, sq2 = (row + 2 * ur) * R + col + 2 * uc;
    if (!attacked_by_team(g, b, other_team, sq1) && !attacked_by_team(g, b, other_team, from))
      push(ml, pack_move(from, sq2, EMPTY, NO_PIECE, rr * R + rc, sq1, r0, r1));
  }
}

/* engine/board.cpp:846-889 GetPseudoLegalMoves2.  The reference iterates piece_list_[turn],
 * whose order is history dependent (SURVEY 8a row 9); here squares are scanned in index order. */
static int pseudo_moves(const Geo *g, const uint8_t *b, uint64_t *out, int cap) {
  MoveList ml = {out, 0, cap};
  int turn = b[g->off_turn] & 3;
  if (b[g->off_king + turn] >= g->nsq) return 0;
  for (int sq = 0; sq < g->nsq; ++sq) {
    uint8_t p = b[sq];
    if (!present(p) || color_of(p) != turn) continue;
    switch (type_of(p)) {
      case PAWN: pawn_moves(g, b, &ml, sq, p); break;
      case KNIGHT: knight_moves(g, b, &ml, sq, p); break;
      case BISHOP: bishop_moves(g, b, &ml, sq, p); break;
      case ROOK: rook_moves(g, b, &ml, sq, p); break;
      case QUEEN: bishop_moves(g, b, &ml, sq, p); rook_moves(g, b, &ml, sq, p); break;
      case KING: king_moves(g, b, &ml, sq, p); break;
    }
  }
  return ml.n;
}

/* engine/board.cpp:1028-1096 MakeMove.  Returns -1 where the reference throws (:1046-1054). */
static int make_move(const Geo *g, uint8_t *b, uint64_t m) {
  int from = MV_FROM(m), to = MV_TO(m), turn = b[g->off_turn] & 3;
  if (from >= g->nsq || to >= g->nsq) return -2; /* off-board: undefined in the reference */
  uint8_t piece = b[from], cap = b[to];
  if (present(cap)) { /* RemovePiece(to) :992-1014 */
    b[to] = EMPTY;
    if (type_of(cap) == KING) b[g->off_king + color_of(cap)] = (uint8_t)g->nsq;
  }
  if (!present(piece)) return -1;
  b[from] = EMPTY;
  if (type_of(piece) == KING) b[g->off_king + color_of(piece)] = (uint8_t)g->nsq;
  int promo = MV_PROMO(m);
  uint8_t placed = promo != NO_PIECE ? mk_piece(turn, promo) : piece; /* :1057-1067 */
  b[to] = placed;
  if (type_of(placed) == KING) b[g->off_king + color_of(placed)] = (uint8_t)to;
  int rf = MV_RFROM(m), rt = MV_RTO(m);
  if (rf < g->nsq && rt < g->nsq) { /* SimpleMove::Present :255 */
    uint8_t rook = b[rf];
    b[rf] = EMPTY;
    if (type_of(rook) == KING && present(rook)) b[g->off_king + color_of(rook)] = (uint8_t)g->nsq;
    b[rt] = rook;
    if (type_of(rook) == KING && present(rook)) b[g->off_king + color_of(rook)] = (uint8_t)rt;
  }
  if (MV_R1(m) & 0x80) b[g->off_rights + turn] = MV_R1(m); /* :1080-1084 */
  b[g->off_turn] = (uint8_t)((turn + 1) & 3);              /* :1088, :1299-1313 */
  return 0;
}

/* src/cpp/board.cpp:59-68 IsKingSafeAfterMove, on a scratch copy instead of make/undo. */
static int king_safe_after(const Geo *g, const uint8_t *b, uint64_t m) {
  uint8_t tmp[256];
  memcpy(tmp, b, (size_t)g->rec);
  int me = b[g->off_turn] & 3;
  if (make_move(g, tmp, m) != 0) return 0;
  int ksq = tmp[g->off_king + me];
  if (ksq >= g->nsq) return 1; /* engine/board.cpp:945-948 */
  return !attacked_by_team(g, tmp, 1 - team_of_color(me), ksq);
}

/* src/cpp/move.cpp:13-16, 63-104: (dx,dy) -> action plane; -1 where GetIndex throws. */
static int action_plane(int R, int dx, int dy) {
  static const int qd[8][2] = {{0, -1}, {-1, -1}, {-1, 0}, {-1, 1}, {0, 1}, {1, 1}, {1, 0}, {1, -1}};
  static const int kd[8][2] = {{-2, -1}, {-2, 1}, {-1, -2}, {-1, 2}, {1, -2}, {1, 2}, {2, -1}, {2, 1}};
  for (int i = 0; i < 8; ++i)
    for (int dist = 1; dist <= R - 1; ++dist)
      if (dx == qd[i][0] * dist && dy == qd[i][1] * dist) return i * (R - 1) + dist - 1;
  for (int i = 0; i < 8; ++i)
    if (dx == kd[i][0] && dy == kd[i][1]) return 8 * (R - 1) + i;
  return -1;
}

static int flat_index(int R, uint64_t m) {
  int from = MV_FROM(m), to = MV_TO(m);
  int pl = action_plane(R, to % R - from % R, to / R - from / R);
  if (pl < 0) return -1;
  return pl * R * R + (from / R) * R + from % R; /* move.cpp:100-104 */
}

static int cmp_key(const void *a, const void *b) {
  const uint64_t *x = (const uint64_t *)a, *y = (const uint64_t *)b;
  return (x[0] > y[0]) - (x[0] < y[0]);
}

/* The legal subset of pseudo[0 .. n-1] in canonical order (ascending flat action index, then promotion type);
 * keyed has room for n entries.  Returns the legal count, writes at most cap moves. */
static int legal_subset(const Geo *g, const uint8_t *b, const uint64_t *pseudo, int n, uint64_t (*keyed)[2],
                        uint64_t *out, int cap) {
  int k = 0;
  for (int i = 0; i < n; ++i)
    if (king_safe_after(g, b, pseudo[i])) {
      keyed[k][0] = (uint64_t)flat_index(g->R, pseudo[i]) * 8 + (uint64_t)MV_PROMO(pseudo[i]);
      keyed[k][1] = pseudo[i];
      ++k;
    }
  qsort(keyed, (size_t)k, sizeof keyed[0], cmp_key);
  for (int i = 0; i < k && i < cap; ++i) out[i] = keyed[i][1];
  return k;
}

/* src/cpp/board.cpp:94-118 GetLegalMoves, returned in canonical order. */
static int legal_moves(const Geo *g, const uint8_t *b, uint64_t *out, int cap) {
  uint64_t pseudo[MAX_MOVES], keyed[MAX_MOVES][2];
  int n = pseudo_moves(g, b, pseudo, MAX_MOVES);
  if (n > MAX_MOVES) abort(); /* engine/board.h:482-486 */
  return legal_subset(g, b, pseudo, n, keyed, out, cap);
}

/* engine/board.cpp:891-939 GetGameResult under the order-independent contract of SURVEY 8a
 * row 8: branches (i) and (iii) exactly; branch (ii) reports IN_PROGRESS and sets
 * *can_capture_king when some legal move takes a king. */
static int game_result(const Geo *g, const uint8_t *b, int *n_legal_out, int *can_capture_king) {
  uint64_t legal[MAX_MOVES];
  int turn = b[g->off_turn] & 3, ry = team_of_color(turn) == 0;
  int n = legal_moves(g, b, legal, MAX_MOVES), kc = 0;
  for (int i = 0; i < n; ++i)
    if (present(MV_CAP(legal[i])) && type_of(MV_CAP(legal[i])) == KING) kc = 1;
  if (n_legal_out) *n_legal_out = n;
  if (can_capture_king) *can_capture_king = kc;
  if (b[g->off_king + turn] >= g->nsq) return ry ? WIN_BG : WIN_RY;
  if (n > 0) return IN_PROGRESS;
  if (!attacked_by_team(g, b, 1 - team_of_color(turn), b[g->off_king + turn])) return STALEMATE;
  return ry ? WIN_BG : WIN_RY;
}

static uint64_t mix(uint64_t seed, uint64_t game, uint64_t ply) {
  uint64_t z = seed ^ (game * 0x9E3779B97F4A7C15ULL) ^ (ply * 0xBF58476D1CE4E5B9ULL);
  z += 0x9E3779B97F4A7C15ULL;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}

static uint64_t perft(const Geo *g, const uint8_t *b, int depth) {
  uint64_t legal[MAX_MOVES];
  int n = legal_moves(g, b, legal, MAX_MOVES);
  if (depth <= 1) return (uint64_t)n;
  uint64_t total = 0;
  uint8_t child[256];
  for (int i = 0; i < n; ++i) {
    memcpy(child, b, (size_t)g->rec);
    make_move(g, child, legal[i]);
    total += perft(g, child, depth - 1);
  }
  return total;
}

/* ------------------------------------------------------------------ C-ABI ---------------- */

int fpo_record_bytes(int R) { return geo(R, 0).rec; }
int fpo_is_legal_location(int R, int IA, int row, int col) {
  Geo g = geo(R, IA);
  return legal_loc(&g, row, col);
}
int fpo_pseudo_moves(int R, int IA, const uint8_t *rec, uint64_t *out, int cap) {
  Geo g = geo(R, IA);
  return pseudo_moves(&g, rec, out, cap);
}
int fpo_legal_moves(int R, int IA, const uint8_t *rec, uint64_t *out, int cap) {
  Geo g = geo(R, IA);
  return legal_moves(&g, rec, out, cap);
}
/* fpo_legal_moves without the reference's 300-move buffer: the full canonical legal list of a crowded position (the
 * reference aborts above 300 pseudo-legal moves; the device rules kernel counts legal moves only).  *n_pseudo = the
 * pseudo-legal count.  Returns the legal count (at most cap moves written), or -1 above WIDE_MOVES pseudo-legal moves. */
#define WIDE_MOVES 1024
int fpo_legal_moves_wide(int R, int IA, const uint8_t *rec, uint64_t *out, int cap, int *n_pseudo) {
  uint64_t pseudo[WIDE_MOVES], keyed[WIDE_MOVES][2];
  Geo g = geo(R, IA);
  int n = pseudo_moves(&g, rec, pseudo, WIDE_MOVES);
  if (n_pseudo) *n_pseudo = n;
  if (n > WIDE_MOVES) return -1;
  return legal_subset(&g, rec, pseudo, n, keyed, out, cap);
}
int fpo_is_attacked_by_team(int R, int IA, const uint8_t *rec, int team, int sq) {
  Geo g = geo(R, IA);
  return attacked_by_team(&g, rec, team, sq);
}
/* fpchess::Board::IsAttackedByPlayer (src/cpp/board.cpp:142-209), the viewer's query.  Its "isLegalPosition" is
 * BoardLocation::Present(), i.e. inside the R x R index range: rays run through the cut corners. */
static int attacked_by_player(const Geo *g, const uint8_t *b, int sq, int color) {
  static const int D8[8][2] = {{1, 0}, {0, 1}, {-1, 0}, {0, -1}, {1, 1}, {1, -1}, {-1, 1}, {-1, -1}};
  static const int KN[8][2] = {{1, 2}, {2, 1}, {-1, -2}, {-2, -1}, {1, -2}, {2, -1}, {-1, 2}, {-2, 1}};
  int R = g->R, lr = sq / R, lc = sq % R;
  /* pawns (:153-162): a pawn of that colour on a neighbour that PawnAttacks (engine/board.cpp:583-604) the square */
  for (int d = 0; d < 8; ++d) {
    int r = lr + D8[d][0], c = lc + D8[d][1];
    if (r < 0 || r >= R || c < 0 || c >= R) continue;
    uint8_t p = b[r * R + c];
    if (color_of(p) == color && type_of(p) == PAWN) {
      int rd = lr - r, cd = lc - c, a = 0;
      switch (color) {
        case RED: a = rd == -1 && abs(cd) == 1; break;
        case BLUE: a = cd == 1 && abs(rd) == 1; break;
        case YELLOW: a = rd == 1 && abs(cd) == 1; break;
        case GREEN: a = cd == -1 && abs(rd) == 1; break;
      }
      if (a) return 1;
    }
  }
  /* knights (:165-171) */
  for (int d = 0; d < 8; ++d) {
    int r = lr + KN[d][0], c = lc + KN[d][1];
    if (r < 0 || r >= R || c < 0 || c >= R) continue;
    uint8_t p = b[r * R + c];
    if (color_of(p) == color && type_of(p) == KNIGHT) return 1;
  }
  /* bishops, rooks, queens (:174-199): the first piece on a ray decides */
  for (int d = 0; d < 8; ++d) {
    int dr = D8[d][0], dc = D8[d][1], r = lr + dr, c = lc + dc;
    for (; r >= 0 && r < R && c >= 0 && c < R; r += dr, c += dc) {
      uint8_t p = b[r * R + c];
      if (!present(p)) continue;
      if (color_of(p) != color) break;
      int t = type_of(p);
      if (t != BISHOP && t != ROOK && t != QUEEN) break;
      if (t == BISHOP && (dr == 0 || dc == 0)) break;
      if (t == ROOK && dr != 0 && dc != 0) break;
      return 1;
    }
  }
  /* kings (:202-207) */
  for (int d = 0; d < 8; ++d) {
    int r = lr + D8[d][0], c = lc + D8[d][1];
    if (r < 0 || r >= R || c < 0 || c >= R) continue;
    uint8_t p = b[r * R + c];
    if (color_of(p) == color && type_of(p) == KING) return 1;
  }
  return 0;
}
int fpo_is_attacked_by_player(int R, int IA, const uint8_t *rec, int sq, int color) {
  Geo g = geo(R, IA);
  return attacked_by_player(&g, rec, sq, color);
}
/* the byte map of fpc_attack_maps (include/fpc.h): bit c = IsAttackedByPlayer(colour c), bit 4+t = IsAttackedByTeam(t),
 * for every square of the R x R box (GetAttackedSquaresPlayers / Teams, src/cpp/board.cpp:120-140, 211-232) */
void fpo_attack_map(int R, int IA, const uint8_t *rec, uint8_t *out) {
  Geo g = geo(R, IA);
  for (int sq = 0; sq < g.nsq; ++sq) {
    int bits = 0;
    for (int c = 0; c < 4; ++c) bits |= attacked_by_player(&g, rec, sq, c) << c;
    for (int t = 0; t < 2; ++t) bits |= attacked_by_team(&g, rec, t, sq) << (4 + t);
    out[sq] = (uint8_t)bits;
  }
}
int fpo_king_in_check(int R, int IA, const uint8_t *rec, int color) {
  Geo g = geo(R, IA);
  int k = rec[g.off_king + color];
  if (k >= g.nsq) return 0;
  return attacked_by_team(&g, rec, 1 - team_of_color(color), k);
}
int fpo_make_move(int R, int IA, const uint8_t *rec, uint64_t move, uint8_t *out) {
  Geo g = geo(R, IA);
  memcpy(out, rec, (size_t)g.rec);
  return make_move(&g, out, move);
}
/* src/cpp/move.cpp:41-61 Move(int flat_index): only from/to are set. */
uint64_t fpo_move_from_flat(int R, int flat) {
  static const int qd[8][2] = {{0, -1}, {-1, -1}, {-1, 0}, {-1, 1}, {0, 1}, {1, 1}, {1, 0}, {1, -1}};
  static const int kd[8][2] = {{-2, -1}, {-2, 1}, {-1, -2}, {-1, 2}, {1, -2}, {1, 2}, {2, -1}, {2, 1}};
  int nsq = R * R, type = flat / nsq, pos = flat % nsq, row = pos / R, col = pos % R, dr, dc;
  if (type < 8 * (R - 1)) {
    int dir = type / (R - 1), dist = type % (R - 1);
    dc = qd[dir][0] * (dist + 1);
    dr = qd[dir][1] * (dist + 1);
  } else {
    int k = type - 8 * (R - 1);
    if (k > 7) k = 7; /* planes past 8(R-1)+7 index out of range in the reference */
    dc = kd[k][0];
    dr = kd[k][1];
  }
  int tr = row + dr, tc = col + dc;
  int to = (tr < 0 || tr >= R || tc < 0 || tc >= R) ? nsq : tr * R + tc;
  return pack_move(pos, to, EMPTY, NO_PIECE, nsq, nsq, 0, 0);
}
int fpo_make_index(int R, int IA, const uint8_t *rec, int flat, uint8_t *out) {
  return fpo_make_move(R, IA, rec, fpo_move_from_flat(R, flat), out);
}
int fpo_move_flat_index(int R, uint64_t move) { return flat_index(R, move); }
int fpo_game_result(int R, int IA, const uint8_t *rec, int *n_legal, int *can_capture_king) {
  Geo g = geo(R, IA);
  return game_result(&g, rec, n_legal, can_capture_king);
}
/* engine/board.cpp:1263-1292 CalculateHeuristic */
int fpo_heuristic(int R, int IA, const uint8_t *rec, int team) {
  static const int val[6] = {1, 3, 3, 5, 9, 0};
  Geo g = geo(R, IA);
  int h = 0;
  for (int sq = 0; sq < g.nsq; ++sq) {
    uint8_t p = rec[sq];
    if (!present(p) || type_of(p) == KING) continue;
    h += team_of(p) == team ? val[type_of(p)] : -val[type_of(p)];
  }
  return h;
}
uint64_t fpo_perft(int R, int IA, const uint8_t *rec, int depth) {
  Geo g = geo(R, IA);
  return perft(&g, rec, depth);
}
uint64_t fpo_mix(uint64_t seed, uint64_t game, uint64_t ply) { return mix(seed, game, ply); }

/* src/cpp/board.cpp:305-356 GetEncodedStates.  out[b][ch][row][col] = 1 with
 * ch = ((color - turn) mod 4)*6 + type - 1, where -1 wraps to 23 (torch negative index, :336),
 * then rot90 by k[b] quarter turns on the last two dims (:354-355; torch.rot90 k=1 sends
 * (r,c) -> (R-1-c, r)).  The reference rotates the whole batch by the colour of states[0];
 * callers reproduce that by passing k[b] = colour(states[0]) for every b. */
void fpo_encode(int R, const uint8_t *recs, int n, const int32_t *k, float *out) {
  Geo g = geo(R, 0);
  memset(out, 0, sizeof(float) * (size_t)n * 24 * (size_t)g.nsq);
  for (int b = 0; b < n; ++b) {
    const uint8_t *rec = recs + (size_t)b * g.rec;
    int turn = rec[g.off_turn] & 3, rot = ((k[b] % 4) + 4) % 4;
    for (int sq = 0; sq < g.nsq; ++sq) {
      uint8_t p = rec[sq];
      if (!present(p)) continue;
      int ch = ((color_of(p) - turn + 4) % 4) * 6 + type_of(p) - 1;
      if (ch < 0) ch += 24;
      int r = sq / R, c = sq % R;
      for (int t = 0; t < rot; ++t) {
        int nr = R - 1 - c, nc = r;
        r = nr;
        c = nc;
      }
      out[((size_t)b * 24 + (size_t)ch) * g.nsq + (size_t)r * R + c] = 1.0f;
    }
  }
}

/* src/py/four_player_chess_board.py:36-55 get_legal_moves_mask with
 * src/cpp/board.cpp:424-449 GetLegalMovesIndices: mask[b][plane][from_row][from_col] = 1,
 * absolute coordinates (no rotation). */
void fpo_mask(int R, int IA, const uint8_t *recs, int n, float *out) {
  Geo g = geo(R, IA);
  size_t per = (size_t)(8 * R + 8) * g.nsq;
  memset(out, 0, sizeof(float) * (size_t)n * per);
  uint64_t legal[MAX_MOVES];
  for (int b = 0; b < n; ++b) {
    int m = legal_moves(&g, recs + (size_t)b * g.rec, legal, MAX_MOVES);
    for (int i = 0; i < m; ++i) out[(size_t)b * per + (size_t)flat_index(R, legal[i])] = 1.0f;
  }
}

/* One ply of the deterministic random playout (SURVEY 8d config 2): canonical legal list,
 * pick = ((mix(seed, game, ply) >> 32) * n) >> 32, make(full).  Returns the result of the
 * position in rec (before the move); writes the successor to out when IN_PROGRESS. */
int fpo_playout_step(int R, int IA, const uint8_t *rec, uint64_t seed, uint64_t game, uint64_t ply, uint8_t *out,
                     int *n_legal, uint64_t *move) {
  Geo g = geo(R, IA);
  uint64_t legal[MAX_MOVES];
  int n = 0, kc = 0;
  int res = game_result(&g, rec, &n, &kc);
  legal_moves(&g, rec, legal, MAX_MOVES);
  if (n_legal) *n_legal = n;
  memcpy(out, rec, (size_t)g.rec);
  if (move) *move = 0;
  if (res != IN_PROGRESS) return res;
  uint32_t pick = (uint32_t)(((mix(seed, game, ply) >> 32) * (uint64_t)n) >> 32);
  if (move) *move = legal[pick];
  make_move(&g, out, legal[pick]);
  return res;
}

/* CPU baseline ("port"): single-thread playouts for >= min_positions positions. */
uint64_t fpo_bench_playout(int R, int IA, const uint8_t *start, uint64_t seed, uint64_t first_game,
                           uint64_t min_positions, int max_plies, uint64_t *checksum) {
  Geo g = geo(R, IA);
  uint64_t positions = 0, sum = 0, game = first_game;
  uint8_t cur[256], nxt[256];
  while (positions < min_positions) {
    memcpy(cur, start, (size_t)g.rec);
    for (int p = 0; p < max_plies; ++p) {
      int n = 0;
      int res = fpo_playout_step(R, IA, cur, seed, game, (uint64_t)p, nxt, &n, NULL);
      ++positions;
      sum += (uint64_t)n * 4 + (uint64_t)res;
      if (res != IN_PROGRESS) break;
      memcpy(cur, nxt, (size_t)g.rec);
    }
    ++game;
  }
  if (checksum) *checksum = sum;
  return positions;
}

/* ------------------------------------------------------------------ PUCT ----------------- */
/* Order-independent checksum over whole playouts of games first_game .. first_game + n_games - 1: the sum over
 * every visited position of  n_legal*4 + result + ((move * 0x9E3779B97F4A7C15) >> 40),  move = the move played
 * (0 where the game ended).  The -m gpu soak test recomputes it from the device's per-step outputs. */
uint64_t fpo_playout_checksum(int R, int IA, const uint8_t *start, uint64_t seed, uint64_t first_game, int n_games,
                              int max_plies, uint64_t *positions_out) {
  Geo g = geo(R, IA);
  uint64_t positions = 0, sum = 0;
  uint8_t cur[256], nxt[256];
  for (int i = 0; i < n_games; ++i) {
    memcpy(cur, start, (size_t)g.rec);
    for (int p = 0; p < max_plies; ++p) {
      int n = 0;
      uint64_t mv = 0;
      int res = fpo_playout_step(R, IA, cur, seed, first_game + (uint64_t)i, (uint64_t)p, nxt, &n, &mv);
      ++positions;
      sum += (uint64_t)n * 4 + (uint64_t)res + ((mv * 0x9E3779B97F4A7C15ull) >> 40);
      if (res != IN_PROGRESS) break;
      memcpy(cur, nxt, (size_t)g.rec);
    }
  }
  if (positions_out) *positions_out = positions;
  return sum;
}

/* src/cpp/node.{h,cpp}: a tree of nodes over one game, children stored contiguously.
 * Arrays are caller-owned (numpy); node 0 is the root (visit_count 1, src/py/mcts.py:30). */
typedef struct {
  int32_t *parent, *first_child, *n_children, *visits, *move;
  double *value_sum, *prior;
} Tree;

/* src/cpp/node.cpp:49-78 SelectChild: argmax of Q + C*sqrt(ln(sqrt(N))/(1+n))*P, first max wins;
 * -1 where the reference throws (no child beats -inf, e.g. NaN scores). */
int fpo_select_child(const int32_t *first_child, const int32_t *n_children, const int32_t *visits,
                     const double *value_sum, const double *prior, int node, double C) {
  int best = -1;
  double best_ucb = -INFINITY;
  double lg = log(sqrt((double)visits[node]));
  for (int i = 0; i < n_children[node]; ++i) {
    int ch = first_child[node] + i;
    int n = visits[ch];
    double q = n > 0 ? value_sum[ch] / n : 0.0;
    double ucb = q + C * sqrt(lg / (1 + n)) * prior[ch];
    if (ucb > best_ucb) {
      best = ch;
      best_ucb = ucb;
    }
  }
  return best;
}

/* src/cpp/node.cpp:133-142 Backpropagate */
void fpo_backpropagate(const int32_t *parent, int32_t *visits, double *value_sum, int node, float value) {
  float v = value;
  while (node >= 0) {
    value_sum[node] += v;
    visits[node] += 1;
    v = -v;
    node = parent[node];
  }
}
