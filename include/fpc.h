/* fpc.h -- C-ABI of the B200-native batched four-player-chess environment.
 *
 * This is the drop-in boundary underneath the reference's pybind11 module `alphazero_cpp`
 * (/root/reference/src/cpp/wrapper.cpp:15-254).  Every entry point names the reference
 * interface it replaces.  Plain pointers and sizes only; no torch types; no exceptions cross
 * this ABI: functions return FPC_OK or a negative code and fpc_last_error() holds the text
 * (the binding turns codes into RuntimeError, wrapper.cpp:17-27).
 *
 * All `d_` pointers are DEVICE pointers on the current CUDA device; `h_` pointers are HOST
 * pointers.  `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); calls
 * taking a stream are asynchronous with respect to the host.  There is NO CPU fallback: with no
 * usable CUDA device every compute entry point fails with FPC_ERR_CUDA.
 *
 * Geometry.  The reference fixes the board at compile time (engine/board.h:22-24).  Here the
 * side length R selects a compiled instantiation: R=14 (invalid_area 3, the 4pchess board of
 * BASELINE.json), R=8 (invalid_area 2, the reference as checked in), R=10 (2), R=13 (3).
 *
 * Board record (one game), fpc_record_bytes(R) bytes, 16-byte aligned in arrays:
 *   [0, R*R)      piece bytes, row-major, the reference's Piece bits (engine/board.h:101-104):
 *                 present<<7 | color<<5 | type<<2; empty = 0x18
 *   [R*R]         side to move (0 RED, 1 BLUE, 2 YELLOW, 3 GREEN)
 *   [R*R+1, +5)   castling rights per colour (engine/board.h:290-291): 0x80 | ks<<6 | qs<<5
 *   [R*R+5, +9)   king square per colour (row*R+col; R*R = captured).  Output only: kernels
 *                 recompute it from the squares.
 *   rest          zero padding.   R=14: 208 B, R=8: 80 B.
 *
 * Move: the reference's 8-byte chess::Move image (engine/board.h:419-435) as a little-endian
 * uint64: byte0 from, byte1 to, byte2 captured Piece bits (0x18 none), byte3 promotion type
 * (6 none), byte4/5 rook from/to (R*R none), byte6 rights before, byte7 rights after (0 absent).
 *
 * Canonical move order.  The reference's move order depends on call history (SURVEY 8a row 9);
 * every list returned here is sorted by (flat action index, promotion type).
 */
#ifndef FPC_H_
#define FPC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FPC_MAX_MOVES 300 /* engine/board.h:706 move_buffer_size_ */
#define FPC_NUM_STATE_CHANNELS 24 /* src/cpp/board.h:21 */

#define FPC_OK 0
#define FPC_ERR_ARG (-1)      /* bad argument (unsupported R, null pointer, negative n) */
#define FPC_ERR_CUDA (-2)     /* CUDA runtime error, or no device */
#define FPC_ERR_MOVE (-3)     /* "piece missing for move" (engine/board.cpp:1046-1054) */
#define FPC_ERR_OVERFLOW (-4) /* more than FPC_MAX_MOVES pseudo-legal moves (reference aborts) */

/* status word written per game by fpc_observe / fpc_playout_step */
#define FPC_STATUS_RESULT_MASK 0x3     /* GameResult: 0 IN_PROGRESS 1 WIN_RY 2 WIN_BG 3 STALEMATE */
#define FPC_STATUS_IN_CHECK 0x100      /* side to move is in check (set only when it has no legal move) */
#define FPC_STATUS_CAN_TAKE_KING 0x200 /* some legal move captures a king (SURVEY 8a row 8) */
#define FPC_STATUS_OVERFLOW 0x400      /* move buffer overflow */
#define FPC_STATUS_FINISHED 0x800      /* playout only: the game in this slot ended and was re-seeded */
#define FPC_STATUS_CHECK 0x1000        /* side to move is in check (engine/board.cpp:941-960), legal moves or not */

const char *fpc_last_error(void);
int fpc_version(void);

/* statics of fpchess::Board (src/cpp/board.cpp:9-14, wrapper.cpp:175-180) */
int fpc_supported(int R);           /* 1 if R is a compiled geometry */
int fpc_invalid_area(int R);        /* Board::invalidArea */
int fpc_record_bytes(int R);
int fpc_num_action_channels(int R); /* Board::num_action_channels = 8R+8 */
int fpc_action_space_size(int R);   /* Board::action_space_size */
int fpc_state_space_size(int R);    /* Board::state_space_size = 24*R*R */

/* fpchess::Move index map (src/cpp/move.cpp:23-104): host-side, no device needed. */
uint64_t fpc_move_from_flat(int R, int flat_index); /* Move(int flat_index), move.cpp:41-61 */
int fpc_move_flat_index(int R, uint64_t move);      /* Move::GetFlatIndex, -1 where GetIndex throws */

/* FEN -> board record (host-side, no device needed): the 4pchess-style FEN of src/py/start_fens.py as
 * src/py/fen_parser.py:104-170 parses it -- fields split on '-': field 0 the side to move (R/B/Y/G), fields 2 / 3
 * kingside / queenside castling availability "a,b,c,d" in colour order, last field the placement (rows split on
 * '/', cells on ','; "rP" = red pawn ..., "x" = one skipped cell, an integer = that many empty cells).  The
 * reference's Python path computes the castling rights and then drops them (fen_parser.py:137-140,170):
 * honour_castling = 0 reproduces that (all rights off), 1 keeps the FEN's rights.  h_record receives
 * fpc_record_bytes(R) bytes.  Returns FPC_ERR_ARG with the parser's message in fpc_last_error() on bad input. */
int fpc_record_from_fen(int R, const char *fen, int honour_castling, uint8_t *h_record);

/* ---- device-pointer batch operations ------------------------------------------------------ */

/* Observation of a batch (rules_kernel, plus expand_kernel when a dense tensor is asked for; FPC_FLAG_INCREMENTAL is
 * ignored here -- it needs a handle, see fpc_observe_tracked).  d_planes / d_mask
 * must be 16-byte aligned.  For each of n board records:
 *   legal moves      = fpchess::Board::GetLegalMoves (src/cpp/board.cpp:94-118) over
 *                      chess::Board::GetPseudoLegalMoves2 (engine/board.cpp:846-889)
 *   status           = chess::Board::GetGameResult (engine/board.cpp:891-939), order-independent
 *                      contract, plus the FPC_STATUS_* flags
 *   planes           = Board::GetEncodedStates (src/cpp/board.cpp:305-356): [n][24][R][R] f32,
 *                      rotated by k quarter turns (d_k[g] if d_k != NULL, else k_all; k_all = -1
 *                      means "each game by its own side to move")
 *   mask             = FourPlayerChess.get_legal_moves_mask
 *                      (src/py/four_player_chess_board.py:36-55): [n][8R+8][R][R] f32, unrotated
 *   flat indices     = Board::GetLegalMovesIndices (src/cpp/board.cpp:424-449) as flat indices
 * Any output pointer may be NULL.  d_moves / d_flat are [n][FPC_MAX_MOVES]. */
int fpc_observe(int R, const uint8_t *d_boards, int n, uint64_t *d_moves, int32_t *d_flat, int32_t *d_counts,
                int32_t *d_status, float *d_planes, const int32_t *d_k, int k_all, float *d_mask, int flags,
                void *stream);

/* Dense outputs and streams.  The compact results (moves, counts, status, boards) are written by
 * rules_kernel on `stream`.  The dense f32 planes / mask are written by expand_kernel on an
 * internal second stream as soon as the rules kernel has produced the records of their ones; by default
 * `stream` then waits for it, so everything is ordered on `stream` as usual.  With
 * FPC_FLAG_ASYNC_DENSE that wait is left out: the next call's rules kernel overlaps this call's
 * expansion (the HBM-bound part), and the caller orders a consumer of the dense tensors with
 * fpc_join(consumer_stream).  State is per host thread and device. */
#define FPC_FLAG_ASYNC_DENSE 1
int fpc_join(void *stream);

/* FPC_FLAG_INCREMENTAL: resident dense tensors updated in place.  A fpc_dense_track handle owns the record of the
 * cells the latest dense call THROUGH IT set to 1.0 in one planes tensor and / or one mask tensor (created for a
 * board size and batch size on the current device).  When a *_tracked call carries this flag and the handle knows
 * the content of every tensor the call asks for, the rules kernel clears the previously set cells and sets the
 * new ones -- some 120 scattered 4-byte stores per game instead of rewriting 113 KB -- and no expansion runs.
 * The result is bit-identical to a full rewrite PROVIDED nothing else wrote to the tensors since the previous call
 * through the handle; the caller declares any such write with fpc_dense_track_invalidate().  Otherwise (first use,
 * another tensor pointer, after an invalidate, no handle) the call does the full rewrite.  Nothing is inferred from
 * pointer identity alone: a handle only vouches for tensors it has itself written since it was created or
 * invalidated, so a tensor freed and re-allocated at the same address must come with a new (or invalidated) handle.
 * Calls through one handle must be issued on one stream, or ordered by the caller.  Everything is ordered on `stream`. */
#define FPC_FLAG_INCREMENTAL 2
typedef struct fpc_dense_track fpc_dense_track;
fpc_dense_track *fpc_dense_track_create(int R, int n); /* NULL on failure (fpc_last_error) */
void fpc_dense_track_invalidate(fpc_dense_track *track);
void fpc_dense_track_destroy(fpc_dense_track *track);   /* waits for the device; NULL is allowed */
/* fpc_observe / fpc_playout_step (below) with a handle; track == NULL is the plain call. */
int fpc_observe_tracked(fpc_dense_track *track, int R, const uint8_t *d_boards, int n, uint64_t *d_moves, int32_t *d_flat,
                        int32_t *d_counts, int32_t *d_status, float *d_planes, const int32_t *d_k, int k_all, float *d_mask,
                        int flags, void *stream);
int fpc_playout_step_tracked(fpc_dense_track *track, int R, uint8_t *d_boards, int n, uint64_t seed, uint64_t *d_game,
                             int32_t *d_ply, const uint8_t *d_start, int max_plies, uint64_t game_stride, uint64_t *d_chosen,
                             int32_t *d_counts, int32_t *d_status, float *d_planes, const int32_t *d_k, int k_all,
                             float *d_mask, uint64_t *d_counters, int flags, void *stream);

/* Releases what the calling host thread holds on the current device (internal streams, events, record workspace),
 * after waiting for its pending work.  The next dense call re-creates them. */
int fpc_shutdown(void);

/* Measurement hook: time every expand_kernel and (dense-path) rules_kernel launch with CUDA events on the
 * streams they run on (up to 4096 launches per enable).  fpc_profile_read waits for those streams and
 * returns the number of timed launches and the summed durations in milliseconds.  The instrumentation is not free:
 * four timestamped event records per step drain the two internal streams between launches and lengthen a 74 us step
 * to 79 us (measured on B200, tools/overlap_probe.py FPC_P_NOPROF), so throughput is measured with the hook off. */
int fpc_profile_enable(int on);
int fpc_profile_read(int *launches, double *expand_ms, double *rules_ms);

/* Board::GetEncodedStates alone (no move generation). */
int fpc_encode(int R, const uint8_t *d_boards, int n, const int32_t *d_k, int k_all, float *d_planes,
               int flags, void *stream);

/* chess::Board::MakeMove (engine/board.cpp:1028-1096) with full generator moves, as used by
 * Board::TakeAction (src/cpp/board.cpp:234-239).  d_err[g] = FPC_OK or FPC_ERR_MOVE.
 * d_in == d_out is allowed. */
int fpc_make_moves(int R, const uint8_t *d_in, const uint64_t *d_moves, int n, uint8_t *d_out, int32_t *d_err,
                   void *stream);

/* MakeMove with index-built moves Move(flat_index) (src/cpp/move.cpp:41-61) -- the self-play
 * path (src/cpp/node.cpp:87-92, src/py/alphazero.py:119-121): only from/to, so no promotion,
 * no rook move, no rights update. */
int fpc_make_index(int R, const uint8_t *d_in, const int32_t *d_flat, int n, uint8_t *d_out, int32_t *d_err,
                   void *stream);

/* chess::Board::CalculateHeuristic (engine/board.cpp:1263-1292) for the team to move. */
int fpc_heuristic(int R, const uint8_t *d_boards, int n, int32_t *d_value, void *stream);

/* One ply of the deterministic random playout for every game slot (BASELINE.json configs[1]):
 * observe the position (planes/mask optional, as fpc_observe), then either finish the game
 * (result != IN_PROGRESS, or d_ply[g]+1 == max_plies) and re-seed the slot from h/d start
 * record with game id += game_stride, or play
 * legal[ ((mix(seed, game, ply) >> 32) * n_legal) >> 32 ] with MakeMove(full).
 * d_boards is updated in place.  d_counters (8 x uint64, may be NULL) accumulates:
 * [0] positions, [1] finished games, [2..5] result histogram of finished games (index =
 * GameResult, 0 = ply cap), [6] sum of n_legal, [7] overflow count. */
int fpc_playout_step(int R, uint8_t *d_boards, int n, uint64_t seed, uint64_t *d_game, int32_t *d_ply,
                     const uint8_t *d_start, int max_plies, uint64_t game_stride, uint64_t *d_chosen,
                     int32_t *d_counts, int32_t *d_status, float *d_planes, const int32_t *d_k, int k_all,
                     float *d_mask, uint64_t *d_counters, int flags, void *stream);

/* Viewer queries (src/cpp/board.cpp:120-232; the pygame UI only).  d_out [n][R*R] bytes, one per square in row-major
 * order (every row / column, the cut corners included, as the reference's loops run):
 *   bit c (0..3) = fpchess::Board::IsAttackedByPlayer(square, colour c) (src/cpp/board.cpp:142-209: rays bounded by the
 *                  R x R index range only, so they run through the cut corners; a piece of another colour or a
 *                  non-slider of the same colour blocks)
 *   bit 4 + t    = chess::Board::IsAttackedByTeam(team t, square) (engine/board.cpp:606-786) */
int fpc_attack_maps(int R, const uint8_t *d_boards, int n, uint8_t *d_out, void *stream);

/* ---- batched PUCT: one warp owns one game's tree in HBM ---------------------------------------
 *
 * Replaces fpchess::Node (src/cpp/node.{h,cpp}) driven by MCTS.search / step / expand
 * (src/py/mcts.py:17-89).  The tree of game g lives in slab g of caller-owned device arrays
 * (struct-of-arrays, node_cap entries per game, children of a node contiguous and in ascending flat
 * action index = torch.nonzero order, mcts.py:83-87).  Node 0 is the root.  Boards are materialised
 * only for nodes that were selected as a leaf (board_cap per game; one per simulation plus the
 * root): a child's board is its parent's board + MakeMove(Move(flat_index)) (node.cpp:87-92), made
 * when the child is first reached instead of at expansion -- same boards, fewer copies.
 *
 * One simulation for all games = fpc_tree_select -> network forward on `d_planes` (PyTorch) ->
 * fpc_tree_expand_backup.
 *
 * Invariants of every slab the calls below write (fpc_tree_advance relies on them):
 *   - parent[i] < i for every node but the root: children are appended at n_nodes when their parent is expanded,
 *     so a node has the smallest index of its subtree;
 *   - first_child = 0 and n_children = 0 for a node that is not expanded;
 *   - a node is materialised (board_idx >= 0) before it is expanded, so its board slot is below those of its
 *     descendants; slot 0 is the root's;
 *   - n_boards <= n_nodes <= node_cap.
 */
typedef struct fpc_tree {
  int32_t R, n_games, node_cap, board_cap;
  double C;               /* Node::C (alphazero.py:294) */
  /* per node, [n_games][node_cap] */
  int32_t *parent;        /* -1 for the root */
  int32_t *first_child;   /* index of the first child in the same slab */
  int32_t *n_children;    /* 0 = not expanded (Node::IsExpanded, node.cpp:14-17) */
  int32_t *visits;        /* Node::visit_count */
  int32_t *move_flat;     /* flat action index of Node::move_made */
  int32_t *board_idx;     /* slot in `boards`, -1 = not materialised */
  double *value_sum;      /* Node::value_sum */
  float *prior;           /* Node::prior (a float32 policy value widened to double by the reference) */
  /* per game, [n_games] */
  int32_t *n_nodes, *n_boards;
  int32_t *leaf;          /* node chosen by the last select, -1 = none (root dropped) */
  int32_t *dropped;       /* 1 once a terminal leaf was reached: the root sits out the remaining
                             simulations (mcts.py:22-23) */
  int32_t *error;         /* bit 0 node_cap exceeded, bit 1 board_cap exceeded, bit 2 no child selectable
                             (the reference throws, node.cpp:72-75), bit 3 index-built move failed */
  uint8_t *boards;        /* [n_games][board_cap][record] */
  /* the leaf batch: input of the rules kernel and of the network */
  uint8_t *leaf_boards;   /* [n_games][record] */
  int32_t *leaf_flat;     /* [n_games][FPC_MAX_MOVES] legal flat indices of the leaf, ascending */
  int32_t *leaf_counts;   /* [n_games] */
  int32_t *leaf_status;   /* [n_games] FPC_STATUS_* of the leaf */
  int32_t *k;             /* [n_games] quarter turns the leaf's planes were rotated by */
} fpc_tree;

/* Roots: node 0 of every game = d_root_boards[g], visit_count 1 (mcts.py:30), no children. */
int fpc_tree_reset(const fpc_tree *t, const uint8_t *d_root_boards, void *stream);

/* Tree reuse between moves (outside the reference, which builds a fresh Node per move, mcts.py:28-31): re-root every
 * game's tree on the root child whose move_flat == d_actions[g], in place.  d_root_boards [n_games][record] (16-byte
 * aligned) = the positions after the move, made with the index-built move (fpc_make_index).  The subtree of that child
 * c is kept when c exists, the subtree has at most max_keep_nodes nodes and at most max_keep_boards materialised
 * boards, and c's board (if materialised) is byte-equal to d_root_boards[g].  Then:
 *   - the kept nodes are renumbered in ascending order of their old index (c becomes node 0); children stay
 *     contiguous and in ascending flat order; parent and first_child are remapped; visits, value_sum, prior,
 *     move_flat and n_children are unchanged, except that node 0 gets parent -1, move_flat -1, prior 0 and
 *     board_idx 0;
 *   - the kept boards are compacted in ascending order of their old slot and board_idx is remapped; slot 0 holds
 *     d_root_boards[g];
 *   - n_nodes / n_boards = the kept counts, leaf = -1, dropped = 0, error = 0.
 * Otherwise (action -1, no such child, a limit exceeded, a board mismatch) the game gets a fresh root from
 * d_root_boards[g], exactly as fpc_tree_reset writes it; that is not an error.  d_kept[g] (may be NULL) = the number
 * of nodes carried over, 0 for a fresh root.  node_cap above FPC_TREE_ADVANCE_MAX_NODE_CAP (the old -> new index
 * map lives in node_cap / 4 bytes of shared memory) and negative limits are FPC_ERR_ARG, before any launch. */
#define FPC_TREE_ADVANCE_MAX_NODE_CAP 524288
int fpc_tree_advance(const fpc_tree *t, const int32_t *d_actions, const uint8_t *d_root_boards, int32_t max_keep_nodes,
                     int32_t max_keep_boards, int32_t *d_kept, void *stream);

/* Node::ChooseLeaf (node.cpp:19-47) for every live game: descend with Node::SelectChild
 * (node.cpp:49-78: argmax of Q + C*sqrt(ln(sqrt(N))/(1+n))*P in double, first maximum wins),
 * materialise the leaf's board, run the rules kernel on the leaf batch (legal moves + GetGameResult)
 * and encode it into d_planes [n_games][24][R][R] (Board::GetEncodedStates).  batch_rotation != 0
 * reproduces the reference: every leaf is rotated by the colour of the first live leaf
 * (src/cpp/board.cpp:354-355; the first leaf that is not terminal, as mcts.py:18-26 drops those before encoding);
 * 0 rotates each leaf by its own side to move.  flags + track (may be NULL): FPC_FLAG_INCREMENTAL updates d_planes
 * in place (the network only reads it between two selects), see above. */
int fpc_tree_select(const fpc_tree *t, int batch_rotation, float *d_planes, int flags, fpc_dense_track *track, void *stream);

/* MCTS.step after the network (mcts.py:66-79) + MCTS.expand (mcts.py:82-89) for every game with a
 * leaf: terminal leaf -> Backpropagate(0 | -1) and drop the root (node.cpp:33-43); otherwise
 * softmax(d_logits[g]) -> ParseActionspace (rotate back by the leaf's k) -> * legal mask ->
 * renormalise -> Node::BackpropagateNodes(value) -> one child per non-zero prior (visit_count 1,
 * node.h:28).  d_logits [n_games][A*R*R] f32 in the network's (rotated) frame, d_values [n_games]. */
int fpc_tree_expand_backup(const fpc_tree *t, const float *d_logits, const float *d_values, void *stream);

/* ---- leaf-parallel PUCT: several leaves per game in one network batch, with a virtual loss --------------------------
 *
 * Outside the reference (one leaf per game and simulation, mcts.py:17-43).  Every live game descends L times per batch,
 * one slot after the other; in_flight[x] counts the earlier slots of the current batch whose path went through node x,
 * and a descent sees the effective statistics
 *   N_eff(x) = visits[x] + VL*in_flight[x],   W_eff(x) = value_sum[x] - (double)(VL*in_flight[x])
 * in Node::SelectChild's arithmetic (q = n > 0 ? W_eff(c)/n : 0 with n = N_eff(c); ucb = q +
 * C*sqrt(ln(sqrt(N_eff(x)))/(1+n))*P(c) in double; the first maximum wins).  With in_flight all zero this is
 * fpc_tree_select's arithmetic to the bit, so slot 0 (and every slot at L = 1) selects what fpc_tree_select selects.
 *
 * Selection, game g, slots j = 0 .. L-1 in ascending order (slot s = g*L + j):
 *   - the endpoint e is the first node with n_children == 0.  in_flight[e] > 0: a COLLISION (not evaluated; its slot
 *     is spent without a visit).  Otherwise a LEAF, whose board is materialised as fpc_tree_select does it;
 *   - in_flight += 1 on every node of the root -> e path, e and the root included (collisions too: that is what steers
 *     later slots away);
 *   - a descent error (no selectable child, board_cap, index-built move) sets the error bits of fpc_tree_select and
 *     drops the game; slot j and every later slot of the game are EMPTY and add no marks.  A dropped game's slots are
 *     all EMPTY.
 * Every leaf and collision slot then goes through the rules kernel and the encoder (a collision carries its
 * endpoint's board), into d_planes [n_games*L][24][R][R]: the network sees a static batch, so CUDA graphs work.
 * batch_rotation != 0: k = the side to move of the first LEAF slot (ascending s) whose status is IN_PROGRESS.
 * leaf[g] = the node of slot g*L when it is a LEAF, else -1 (at L = 1 what fpc_tree_select writes).
 *
 * Expand / backup, game g, slots in ascending j (the outputs of COLLISION and EMPTY slots are ignored):
 *   - LEAF, terminal: Backpropagate(0 | -1); the game is dropped after this batch (its later slots still count: they
 *     ran concurrently);
 *   - LEAF, in progress: Backpropagate(value), then one child per non-zero prior appended at n_nodes, the priors
 *     bit-identical to fpc_tree_expand_backup's for the same logits, k and legal list.  The node_cap check is made per
 *     slot against the running n_nodes: a slot that does not fit sets error bit 0 and is backed up without children;
 *   - the f64 additions to any one node's value_sum happen in ascending slot order: the bits of a sequential
 *     slot-by-slot backup;
 *   - afterwards in_flight is zero on every node again, whatever errors occurred.
 * num_searches simulations are num_searches / L batches.  The first batch after a reset reaches the unexpanded root in
 * every slot: one leaf, L-1 collisions.  Arena sizes per batch: at most one new board and one expansion per slot.
 *
 * fpc_tree_reset and fpc_tree_advance do not touch in_flight: the caller zeroes it once and the two calls below keep
 * it zero.  L outside 1 .. FPC_MAX_LEAVES_PER_GAME, virtual_loss < 1, null arrays and misaligned logits are
 * FPC_ERR_ARG, before any launch. */
#define FPC_MAX_LEAVES_PER_GAME 256
#define FPC_SLOT_EMPTY 0
#define FPC_SLOT_LEAF 1
#define FPC_SLOT_COLLISION 2
typedef struct fpc_leaf_batch {
  int32_t L;              /* leaf slots per game and batch */
  int32_t virtual_loss;   /* VL >= 1 */
  int32_t *in_flight;     /* [n_games][node_cap], zero between batches */
  /* per slot, [n_games*L] */
  int32_t *slot_node;     /* the endpoint of the slot's descent, -1 for an EMPTY slot */
  int32_t *slot_kind;     /* FPC_SLOT_* */
  uint8_t *leaf_boards;   /* [n_games*L][record] */
  int32_t *leaf_flat;     /* [n_games*L][FPC_MAX_MOVES] */
  int32_t *leaf_counts;
  int32_t *leaf_status;
  int32_t *k;
  float *priors;          /* [n_games*L][FPC_MAX_MOVES] scratch of fpc_tree_expand_backup_leaves */
  /* per game, [n_games] */
  int32_t *collisions;    /* += the COLLISION slots of every select; the caller zeroes it */
} fpc_leaf_batch;

/* One batch's selection (see above), the rules kernel and the planes; flags + track as in fpc_tree_select (the track
 * handle sized for n_games*L). */
int fpc_tree_select_leaves(const fpc_tree *t, const fpc_leaf_batch *b, int batch_rotation, float *d_planes, int flags,
                           fpc_dense_track *track, void *stream);
/* The batch's expand / backup (see above).  d_logits [n_games*L][A*R*R] f32 (16-byte aligned), d_values [n_games*L]. */
int fpc_tree_expand_backup_leaves(const fpc_tree *t, const fpc_leaf_batch *b, const float *d_logits,
                                  const float *d_values, void *stream);

/* ---- Dirichlet exploration noise at the root ------------------------------------------------------------------------
 *
 * AlphaZero's root noise, outside the reference (its args carry dirichlet_alpha / dirichlet_epsilon, alphazero.py:291-306,
 * and mcts.py:45 defines add_dirichlet_noise, which nothing calls).  For every game g with d_done[g] == 0,
 * dropped[g] == 0 and k = n_children[0] > 0, the root's children c_i = first_child[0] + i, i = 0 .. k-1 (slab order):
 *   gamma_i ~ Gamma(alpha, 1) as below;  eta_i = gamma_i / S with S = sum_i gamma_i in f64 (S == 0, possible only
 *   when every draw underflows at alpha below ~0.05: eta_i = 1/k);
 *   prior[c_i] = (float)((1 - (double)epsilon) * (double)prior[c_i] + (double)epsilon * eta_i);  d_done[g] = 1.
 * Nothing else is written, and games that fail the condition are left exactly as they are, so a second call with the
 * same d_done changes nothing.  The order of the f64 sum is fixed by the kernel (a restatement that sums in another
 * order may differ in the last bits of S).
 *
 * The draws are counter-based: those of game g depend only on (seed, d_keys[g], i), never on g's place in the batch,
 * the launch shape or the GPU.  With mix64 of csrc/fpc_device.cuh, uniform j of child i is, in double arithmetic,
 *   U(i, j) = ((double)(mix64(seed, (uint64_t)d_keys[g], (uint64_t)i << 32 | j) >> 11) + 0.5) * 2^-53   (never 0).
 * Gamma (Marsaglia-Tsang, f64): a = alpha < 1 ? alpha + 1 : alpha, d = a - 1/3, c = 1/sqrt(9d).  Attempt t = 0 .. 63:
 *   x = sqrt(-2 ln U(i, 3t)) * cos(2pi * U(i, 3t+1))  (Box-Muller, 2pi = 6.283185307179586);  v = 1 + c*x;
 *   v <= 0: rejected;  else V = v^3, accepted when ln U(i, 3t+2) < x*x/2 + d - d*V + d*ln V, giving d*V.
 * After 64 rejections the draw is d itself.  For alpha < 1 the result is multiplied by U(i, 192)^(1/alpha).
 *
 * alpha not positive and finite, epsilon outside [0, 1], null d_keys / d_done and a bad tree are FPC_ERR_ARG, before
 * any launch.  d_keys [n_games] i64, d_done [n_games] i32. */
int fpc_tree_root_noise(const fpc_tree *t, uint64_t seed, const int64_t *d_keys, float alpha, float epsilon,
                        int32_t *d_done, void *stream);

/* ---- Gumbel root search: sequential halving and an improved policy ---------------------------------------------------
 *
 * Gumbel AlphaZero's root (Danihelka et al., "Policy improvement by planning with Gumbel", ICLR 2022; mctx's
 * gumbel_muzero_policy), outside the reference.  Only the root's step changes: below it the descent is Node::SelectChild
 * exactly as in fpc_tree_select.  For game g with k = n_children[0] > 0 children c_i = first_child[0] + i, i = 0 .. k-1
 * (slab order), all in f64:
 *   N_i = visits[c_i] - 1 (children are created with visit_count 1), s = sum N_i, Nmax = max N_i;
 *   q_i = value_sum[c_i] / N_i for N_i > 0 (the frame SelectChild maximises at the root);
 *   v = -(s == 0 ? value_sum[0] : root_value[g]): the root's network value in the frame of q_i;
 *   l_i = log p_i - max_j log p_j with p_i = (double)prior[c_i];
 *   g_i = scale * (-log(-log U_i)), U_i = ((double)(mix64(seed, (uint64_t)keys[g], (uint64_t)i << 32 | 2^31) >> 11)
 *         + 0.5) * 2^-53 (the root noise's uniform U(i, j) at j = 2^31, a stream disjoint from its j <= 192);
 *   completed Q (mctx's qtransform_completed_by_mix_value): w_i = max(p_i, 2^-126);
 *         W = (sum_{N_i>0} w_i*q_i) / (sum_{N_i>0} w_i), 0 when no child is visited;
 *         v_mix = (v + s*W) / (1 + s);  cq_i = N_i > 0 ? q_i : v_mix;
 *         r_i = (cq_i - min cq) / max(max cq - min cq, 1e-8);  sigma_i = ((c_visit + Nmax) * c_scale) * r_i;
 *   z_i = l_i + sigma_i;  score_i = max(-1e9, g_i + z_i);
 *   cv(s) = mctx's get_sequence_of_considered_visits(m', n_sims)[s], m' = min(max_considered, k), extended past n_sims:
 *         m' <= 1: s.  Else L2 = ceil(log2 m'), c = m', v = 0; loop: e = max(1, n_sims / (L2*c)) (integer division);
 *         s < e*c: cv = v + s / c; else s -= e*c, v += e, c = max(2, c / 2).
 * Every sum, min and max above runs in one order: child i on lane i % 32, each lane over its children in ascending i,
 * then the 32 lane results combined by the xor butterfly over offsets 16, 8, 4, 2, 1 (x = x + x[lane ^ o]).  No
 * product is fused into a sum.
 *
 * fpc_tree_select_gumbel: fpc_tree_select with this root step.  A game that is dropped gets leaf -1; one whose root is
 * not expanded is selected exactly as fpc_tree_select selects it.  Otherwise, when s == 0, root_value[g] =
 * value_sum[0] (a fresh root holds exactly its network value once its expansion has backed it up); the root's child is
 * c_i for the i maximising score_i over {i : N_i == cv(s)}, the first maximum in ascending i winning, and the descent
 * continues from it with Node::SelectChild, then materialises, observes and encodes the leaf as fpc_tree_select does.
 * While every root visit followed the schedule that set is never empty; if it is, error bit 2 is set and the game
 * dropped, as for a failed SelectChild.  The reference's terminal rule is unchanged: a terminal leaf drops the root for
 * the rest of the search.  Continuing a search past its n_sims follows the extended schedule (c = 2 from then on).
 *
 * fpc_tree_gumbel_result: for every game (dropped ones too: the result comes from the visits they have), with cv = Nmax
 * and the same score, d_action[g] = move_flat of the best child, and d_policy[g][i] = (float)(e_i / E) with
 * e_i = exp(z_i - max_j z_j), E = sum e_i (the order above), 0 for i >= k: softmax(l + sigma), the improved policy.  A
 * game with k == 0 gets action -1 and a zero row.  Nothing else is written.
 *
 * max_considered outside 1 .. FPC_MAX_MOVES, n_sims < 0, scale / c_visit / c_scale negative or not finite, null keys /
 * root_value / d_action / d_policy and a bad tree are FPC_ERR_ARG, before any launch.  keys [n_games] i64, root_value
 * [n_games] f64, d_action [n_games] i32, d_policy [n_games][FPC_MAX_MOVES] f32. */
typedef struct fpc_gumbel {
  uint64_t seed;
  const int64_t *keys;     /* per-game keys of the draws: a game's g_i depend only on (seed, key, i) */
  int32_t max_considered;  /* m, the candidates of the first halving phase */
  int32_t n_sims;          /* simulations the schedule is planned for */
  double scale;            /* Gumbel scale; 0 = a deterministic search */
  double c_visit, c_scale; /* sigma's constants (the paper's 50 and 0.1) */
  double *root_value;      /* [n_games] the root's value_sum when s was 0, written by the select */
} fpc_gumbel;
int fpc_tree_select_gumbel(const fpc_tree *t, const fpc_gumbel *gb, int batch_rotation, float *d_planes, int flags,
                           fpc_dense_track *track, void *stream);
int fpc_tree_gumbel_result(const fpc_tree *t, const fpc_gumbel *gb, int32_t *d_action, float *d_policy, void *stream);

/* ---- Gumbel MuZero interior selection: the completed-Q improved policy below the Gumbel root -------------------------
 *
 * The second half of Gumbel MuZero (Danihelka et al., ICLR 2022; mctx's gumbel_muzero_interior_action_selection), outside
 * the reference.  fpc_tree_select_gumbel_interior is fpc_tree_select_gumbel with its root step unchanged (the halving
 * schedule, the draws, root_value) and this step at every node x the descent passes below the root, with
 * k = n_children[x] > 0 children c_i = first_child[x] + i, i = 0 .. k-1, all in f64:
 *   N_i, s, Nmax, q_i, l_i, w_i, W, v_mix, cq_i, r_i and sigma_i exactly as the root's recipe above states them, with x
 *         in place of the root, the same c_visit / c_scale, and
 *   u = (s == 0 ? value_sum[x] : d_node_value[g][x]), v = -u: x's network value in the frame of q_i.  When s == 0 the
 *         select writes d_node_value[g][x] = value_sum[x]: x gained its children in the expansion that backed its own
 *         network value up, and no descent has passed x since, so value_sum[x] is exactly that value (the root_value
 *         rule, applied to every node);
 *   z_i = l_i + sigma_i;  pi'_i = e_i / E with e_i = exp(z_i - max_j z_j), E = sum e_i (fpc_tree_gumbel_result's
 *         soft-max, in its order, before its cast to f32);
 *   score_i = pi'_i - (double)N_i / (1 + (double)s)  (both quotients rounded, then one rounded subtraction).
 * The child is c_i for the first maximum of score_i in ascending i: no draws and no keys below the root, the step is
 * deterministic.  If no score compares greater than -inf (NaN inputs), error bit 2 is set and the game dropped, as for a
 * failed SelectChild.  Sums, maxima and minima run in the root's order (lane i % 32, lanes ascending, then the xor
 * butterfly 16 .. 1) and no product is fused into a sum.  The terminal rule, the materialisation, the observe and the
 * encode of the leaf are fpc_tree_select's.  fpc_tree_gumbel_result serves this search unchanged: the root's statistics
 * are the same.
 *
 * The caller's contract for d_node_value [n_games][node_cap] f64: every simulation since the tree's reset went through
 * this select.  An entry is then read only after this select wrote it, so the slab needs no initialisation and
 * fpc_tree_reset does not touch it.  Null d_node_value, every refusal of fpc_tree_select_gumbel and a bad tree are
 * FPC_ERR_ARG, before any launch. */
int fpc_tree_select_gumbel_interior(const fpc_tree *t, const fpc_gumbel *gb, double *d_node_value, int batch_rotation,
                                    float *d_planes, int flags, fpc_dense_track *track, void *stream);

/* ---- leaf-parallel Gumbel search: several halving steps per game in one network batch ------------------------------
 *
 * The Gumbel search (root-only, or with the interior step when d_node_value is not NULL) over the leaf batch above:
 * num_searches / L batches of n_games*L network rows, slot s = g*L + j, slot kinds LEAF / COLLISION / EMPTY, committed
 * by fpc_tree_expand_backup_leaves unchanged.  Within one round of a halving phase the schedule visits distinct root
 * children, so those visits share a batch with no virtual loss at the root.  One more per-game array:
 *   d_issued [n_games][FPC_MAX_MOVES] i32: I_i, the LEAF and COLLISION slots that took root child i since the tree's
 *   reset.  At L = 1, and in any batch without collisions, I_i = N_i (visits - 1).  The caller zeroes it whenever it
 *   resets the tree, as it zeroes in_flight once.
 *
 * fpc_tree_select_gumbel_leaves, game g (a dropped game: every slot EMPTY):
 *   1. root not expanded: every slot reaches the root, one LEAF and L-1 COLLISIONs (the leaf batch's first-batch rule);
 *      d_issued is not touched;
 *   2. root expanded: score_i = max(-1e9, g_i + l_i + sigma_i) is computed ONCE per batch from the committed statistics,
 *      exactly as fpc_tree_select_gumbel computes it (N_i, Nmax committed; root_value[g] = value_sum[0] when s == 0).
 *      Then for slots j = 0 .. L-1 in ascending order: t = sum_i I_i, cv(t) from the schedule above planned for
 *      gb->n_sims (a caller plans num_searches - L: the first batch expands the root); the slot's root child is the
 *      first maximum of score_i over {i : I_i == cv(t)}; I_i += 1; the descent continues below that child with the leaf
 *      batch's rule: effective statistics N + VL*in_flight and W - VL*in_flight, an endpoint with in_flight > 0 is a
 *      COLLISION, in_flight += 1 along the whole path, the root included.  The schedule runs on I, not on N, so a
 *      collision only lowers N_i and the candidate set is never empty; if it is anyway, or any later step of the
 *      descent fails, the leaf batch's descent-error rule applies (the error bits of fpc_tree_select, e.g. bit 2; the
 *      game is dropped; this slot and every later one are EMPTY) and the failed slot adds nothing to I;
 *   3. below the root with d_node_value: the interior step of fpc_tree_select_gumbel_interior over the effective
 *      statistics (N_eff, q from W_eff, s_eff, Nmax_eff).  x's network value follows the COMMITTED s = sum (visits - 1)
 *      of x's children: s == 0: u = value_sum[x] and d_node_value[g][x] = value_sum[x] is written; else u =
 *      d_node_value[g][x].  Pending descents do not touch value_sum, so the caching argument above still holds.  Without
 *      d_node_value the descent below the root is Node::SelectChild with virtual loss, as in fpc_tree_select_leaves;
 *   4. the rules kernel, the encoder, batch_rotation, leaf[g] and collisions as in fpc_tree_select_leaves.
 * Sums, maxima and minima run in the Gumbel order (lane i % 32, lanes ascending, then the xor butterfly 16 .. 1) and no
 * product is fused into a sum.  Called at L = 1 this select writes what fpc_tree_select_gumbel (or _interior) writes in
 * every tree array.
 *
 * fpc_tree_gumbel_result_leaves: fpc_tree_gumbel_result's recipe with the survivors {i : I_i == max I} in place of
 * {i : N_i == Nmax}, so a visit lost to a collision cannot demote a survivor; the improved policy softmax(l + sigma)
 * comes from the committed statistics, unchanged.  It equals fpc_tree_gumbel_result whenever I == N.
 *
 * Every refusal of fpc_tree_select_gumbel and of fpc_tree_select_leaves, null d_issued, and for the result null
 * d_action / d_policy are FPC_ERR_ARG, before any launch. */
int fpc_tree_select_gumbel_leaves(const fpc_tree *t, const fpc_gumbel *gb, const fpc_leaf_batch *b, int32_t *d_issued,
                                  double *d_node_value, int batch_rotation, float *d_planes, int flags,
                                  fpc_dense_track *track, void *stream);
int fpc_tree_gumbel_result_leaves(const fpc_tree *t, const fpc_gumbel *gb, const int32_t *d_issued, int32_t *d_action,
                                  float *d_policy, void *stream);

/* ---- Keyed move sampling from the root's visit counts ---------------------------------------------------------------
 *
 * The played move of the reference's self-play (alphazero.py:108-118: probs = visits / sum, probs ** (1/temperature),
 * multinomial), drawn from a counter-based uniform so that a game's move depends only on (seed, d_keys[g]) and its own
 * tree, never on its place in the batch.  For game g with dropped[g] == 0 and k = n_children[0] > 0, the root's children
 * c_i = first_child[0] + i, i = 0 .. k-1 (slab order), with v_i = max(visits[c_i], 0) (the stored counts, including
 * the 1 every child is created with) and V = sum v_i (exact, integer):
 *   temperature == 1:  w_i = (double)v_i (the integers themselves: every sum below is exact);
 *   otherwise:         w_i = pow((double)v_i / (double)V, 1.0 / temperature) in f64;
 *   P_i = P_{i-1} + w_i with P_{-1} = 0, one rounded f64 addition per child in ascending i;  W = P_{k-1};
 *   U = ((double)(mix64(seed, (uint64_t)d_keys[g], 2^31 + 1) >> 11) + 0.5) * 2^-53 (the root noise's uniform U(i, j)
 *       at i = 0, j = SAMPLE_J = 2^31 + 1: a stream disjoint from the noise's j <= 192 and Gumbel's j = 2^31);
 *   t = U * W (one rounded product);
 *   d_action[g] = move_flat[c_i] for the smallest i with P_i > t; if none (t rounded up to W), the largest i with w_i > 0.
 * A game that is dropped, whose root has no children, or whose W is not positive (no visits, or every w_i underflowed)
 * gets d_action[g] = -1.  Nothing but d_action is written.
 *
 * temperature not positive and finite, null d_keys / d_action and a bad tree are FPC_ERR_ARG, before any launch.
 * d_keys [n_games] i64, d_action [n_games] i32. */
int fpc_tree_sample_root(const fpc_tree *t, uint64_t seed, const int64_t *d_keys, double temperature,
                         int32_t *d_action, void *stream);

/* ---- host-buffer operations (per-object calls of the binding; e2e measurement) ------------- */

typedef struct fpc_ctx fpc_ctx;

/* One context per (device, R): a stream plus pinned staging and device buffers for up to
 * max_n boards.  Not thread-safe; one per host thread. */
fpc_ctx *fpc_ctx_create(int device, int R, int max_n);
void fpc_ctx_destroy(fpc_ctx *ctx);
void *fpc_ctx_stream(fpc_ctx *ctx);

/* Host in, host out.  Any output may be NULL.  h_planes / h_mask are host buffers; when the
 * caller wants the tensors left on the device (the reference's device="cuda"), it passes
 * d_planes / d_mask (device pointers) instead and NULL for the host ones. */
int fpc_host_observe(fpc_ctx *ctx, const uint8_t *h_boards, int n, uint64_t *h_moves, int32_t *h_flat,
                     int32_t *h_counts, int32_t *h_status, float *h_planes, float *d_planes, int k_all,
                     float *h_mask, float *d_mask);
int fpc_host_make_moves(fpc_ctx *ctx, const uint8_t *h_in, const uint64_t *h_moves, int n, uint8_t *h_out,
                        int32_t *h_err);
int fpc_host_make_index(fpc_ctx *ctx, const uint8_t *h_in, const int32_t *h_flat, int n, uint8_t *h_out,
                        int32_t *h_err);
/* One playout ply through host buffers: boards, game ids and plies are copied in, stepped and
 * copied back; planes/mask stay on the device (d_planes/d_mask may be NULL).  The call returns when
 * the host buffers hold the results.  With FPC_FLAG_ASYNC_DENSE it does not wait for the dense
 * tensors: their expansion overlaps the next call, and fpc_ctx_sync() waits for it. */
int fpc_host_playout_step(fpc_ctx *ctx, uint8_t *h_boards, int n, uint64_t seed, uint64_t *h_game,
                          int32_t *h_ply, const uint8_t *h_start, int max_plies, uint64_t game_stride,
                          int32_t *h_counts, int32_t *h_status, float *d_planes, int k_all, float *d_mask,
                          int flags);
int fpc_ctx_sync(fpc_ctx *ctx);

/* Run the context's copies and kernels on `stream` (e.g. PyTorch's current stream, when outputs go into tensors that
 * stream's allocator owns) instead of the context's own one; NULL switches back.  Host-buffer calls still return only
 * when their results have landed. */
int fpc_ctx_set_stream(fpc_ctx *ctx, void *stream);
int fpc_current_device(void); /* cudaGetDevice, or a negative code */

/* Page-locked host memory for the h_ buffers above (pageable memory works too, through the driver's staging). */
void *fpc_host_alloc(size_t bytes); /* NULL on failure (fpc_last_error) */
void fpc_host_free(void *p);

/* Node::ExpandNodes (src/cpp/node.cpp:79-131) / Board::TakeAction (src/cpp/board.cpp:234-239) for a batch in ONE trip:
 * child[i] = MakeMove(h_parents[i], h_moves[i]) (full 8-byte moves), and the observation of every child -- status word
 * (GetGameResult + flags) and legal-move count -- so that the binding answers the children's GetGameResult /
 * GetLegalMoves without another trip.  The children's legal moves stay in the context ([n][FPC_MAX_MOVES] on the
 * device) until the next call through it; fpc_host_fetch_moves copies the first `stride` moves of each of the n rows
 * to h_moves [n][stride] (stride = the largest count the caller needs).  h_flat (may be NULL) receives the flat
 * action indices the same way when asked for in fpc_host_fetch_moves. */
int fpc_host_expand(fpc_ctx *ctx, const uint8_t *h_parents, const uint64_t *h_moves, int n, uint8_t *h_children,
                    int32_t *h_err, int32_t *h_counts, int32_t *h_status);
int fpc_host_fetch_moves(fpc_ctx *ctx, int n, int stride, uint64_t *h_moves);
/* Board::GetEncodedStates alone from host records into a device tensor (k_all as in fpc_encode). */
int fpc_host_encode(fpc_ctx *ctx, const uint8_t *h_boards, int n, int k_all, float *d_planes);
int fpc_host_heuristic(fpc_ctx *ctx, const uint8_t *h_boards, int n, int32_t *h_value);
int fpc_host_attack_maps(fpc_ctx *ctx, const uint8_t *h_boards, int n, uint8_t *h_out);

/* ---- environment-owned board store + DLPack (SURVEY 8b) -------------------------------------------------------
 *
 * For consumers that are not PyTorch: the library owns the device memory of n games (board records, per-game
 * observation outputs, the dense planes / mask tensors) and hands any of them out as a DLPack DLManagedTensor
 * (dlpack.h v0.8 layout, restated below so that this header stands alone), zero-copy.  The managed tensor keeps the
 * environment alive: the store is freed when fpc_env_destroy has been called AND every exported tensor's deleter has
 * run.  All work of an environment is ordered on its own stream (fpc_env_stream); fpc_env_sync waits for it. */
typedef struct fpc_env fpc_env;
fpc_env *fpc_env_create(int device, int R, int n); /* NULL on failure (fpc_last_error) */
void fpc_env_destroy(fpc_env *env);
void *fpc_env_stream(fpc_env *env);
int fpc_env_sync(fpc_env *env);
int fpc_env_set_boards(fpc_env *env, const uint8_t *h_boards, int first, int count); /* host records -> store */
int fpc_env_get_boards(fpc_env *env, uint8_t *h_boards, int first, int count);
/* fpc_observe over the store into the environment's own outputs (which = bit set of FPC_ENV_* below) */
int fpc_env_observe(fpc_env *env, int which, int k_all);
/* fpc_playout_step over the store (start record: host pointer), same outputs */
int fpc_env_playout_step(fpc_env *env, uint64_t seed, const uint8_t *h_start, int max_plies, uint64_t game_stride,
                         int which, int k_all);
#define FPC_ENV_BOARDS 1   /* uint8  [n][record]            */
#define FPC_ENV_COUNTS 2   /* int32  [n]                    */
#define FPC_ENV_STATUS 4   /* int32  [n]                    */
#define FPC_ENV_MOVES 8    /* int64  [n][FPC_MAX_MOVES]     */
#define FPC_ENV_FLAT 16    /* int32  [n][FPC_MAX_MOVES]     */
#define FPC_ENV_PLANES 32  /* float32 [n][24][R][R]         */
#define FPC_ENV_MASK 64    /* float32 [n][8R+8][R][R]       */
#define FPC_ENV_PLY 128    /* int32  [n]   (playout)        */
#define FPC_ENV_GAME 256   /* int64  [n]   (playout)        */

/* dlpack.h (v0.8) restated: identical layout, guarded so that a translation unit including the real header first
 * keeps its definitions. */
#ifndef DLPACK_DLPACK_H_
typedef enum { kDLCPU = 1, kDLCUDA = 2, kDLCUDAHost = 3 } DLDeviceType;
typedef struct { DLDeviceType device_type; int32_t device_id; } DLDevice;
typedef enum { kDLInt = 0U, kDLUInt = 1U, kDLFloat = 2U } DLDataTypeCode;
typedef struct { uint8_t code; uint8_t bits; uint16_t lanes; } DLDataType;
typedef struct {
  void *data;
  DLDevice device;
  int32_t ndim;
  DLDataType dtype;
  int64_t *shape;
  int64_t *strides; /* NULL = compact row-major */
  uint64_t byte_offset;
} DLTensor;
typedef struct DLManagedTensor {
  DLTensor dl_tensor;
  void *manager_ctx;
  void (*deleter)(struct DLManagedTensor *self);
} DLManagedTensor;
#endif
/* One of the FPC_ENV_* tensors as a DLManagedTensor (the consumer calls ->deleter when done; wrap it in a PyCapsule
 * named "dltensor" for torch.utils.dlpack.from_dlpack / cupy.from_dlpack).  NULL on failure. */
DLManagedTensor *fpc_env_dlpack(fpc_env *env, int which);

#ifdef __cplusplus
}
#endif
#endif /* FPC_H_ */
