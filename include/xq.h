/* xq.h -- C ABI of the B200-native batched Xiangqi environment + DQN trainer.
 *
 * This is the drop-in boundary for the self-play training path of Qervas/cn_chess_ai.
 * The reference has no FFI/plugin interface: its hot path sits behind four C++ headers
 * (include/chessboard.h, include/action.h, include/chessai.h, include/dqn.h) that
 * MainWindow/Worker consume directly.  Each entry point below names the reference
 * member function(s) it replaces (file:line under /root/reference); the Qt-free C++
 * adapter classes in cn_chess_ai_b200/adapter/ re-expose the original class API
 * (ChessBoard / Action / ChessAI / DQN) on top of these calls.
 *
 * Conventions: extern "C", opaque handles, plain pointers and sizes, int status
 * (0 = XQ_OK); no exception crosses the boundary; xq_last_error() returns the text of
 * the last failure on the calling thread.  Pointers named *_host are host memory, the
 * call copies to/from the device and returns after the result is in the host buffer.
 * Calls are stream-ordered on the handle's stream (xq_env_set_stream / xq_dqn_set_stream).
 * There is no CPU fallback: every compute entry point launches sm_100a kernels and
 * fails with XQ_ERR_CUDA when no device is present.
 */
#ifndef XQ_H
#define XQ_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XQ_ROWS 10
#define XQ_COLS 9
#define XQ_SQUARES 90
#define XQ_STATE_SIZE 1260   /* 90 squares x 14 channels, src/chessai.cpp:268-289,399 */
#define XQ_MAX_ACTIONS 128   /* hard bound of getAllValidActions is 119 (SURVEY A.3) */
#define XQ_MAX_MOVES 200     /* ChessBoard::maxMovePerGame, include/chessboard.h:63 */

enum { XQ_OK = 0, XQ_ERR_INVALID = 1, XQ_ERR_CUDA = 2, XQ_ERR_NOMEM = 3, XQ_ERR_IO = 4, XQ_ERR_STATE = 5 };
enum { XQ_RED = 0, XQ_BLACK = 1, XQ_NONE = 2 };  /* PieceColor, include/chessboard.h:12-14 */

/* Packed environment record: the unit of HBM state, 64 B, 64-B aligned.
 * Replaces ChessBoard's fields (include/chessboard.h:61-64,77-78): QVector<ChessPiece> board,
 * moveCount, currentPlayer, redScore, blackScore.  Square s = row*9+col is nibble (s&7) of
 * sq[s>>3]; code 0 empty, 1..7 Red PieceType (General..Soldier, include/chessboard.h:8-10),
 * 8..14 Black (PieceType+7) = one-hot channel+1 of getStateRepresentation. */
typedef struct {
    uint32_t sq[12];
    uint16_t move_count;
    uint8_t player;       /* 0 Red, 1 Black */
    uint8_t flags;        /* reserved, 0 */
    int32_t red_score;
    int32_t black_score;
    uint32_t ctr;         /* plies applied to this env slot since creation: RNG counter */
} xq_env_rec;

/* Action (include/action.h:4-11) packed as (from<<7)|to, squares 0..89. */
typedef uint16_t xq_action;
#define XQ_ACTION(from, to) ((xq_action)(((from) << 7) | (to)))
#define XQ_ACTION_FROM(a) ((a) >> 7)
#define XQ_ACTION_TO(a) ((a) & 127)
#define XQ_ACTION_NONE 0xFFFF

/* One ply of a traced rollout. */
typedef struct {
    xq_action action;
    uint8_t n_legal;   /* size of the ordered action list the action was drawn from */
    uint8_t flags;     /* bit0 done, bits1-2 winner (PieceColor), bits4-7 captured piece code */
    int32_t reward;    /* ChessAI::evaluateBoard for the mover, src/chessai.cpp:311-345 */
} xq_trace_rec;

typedef struct {
    uint64_t steps, games, red_wins, black_wins, cap_games, captures;
    int64_t reward_sum;
    uint64_t legal_sum;
} xq_env_stats;

typedef struct xq_env_s* xq_env_t;

const char* xq_last_error(void);
const char* xq_version(void);
int xq_device_count(int* count);

/* Counter RNG of the framework (the reference is unseedable: std::srand(time) src/chessai.cpp:13,
 * random_device src/dqn.cu:97).  x = splitmix64-finaliser(seed + env_id*phi + ctr*C);
 * list index draw = x>>33, explore coin = x & 0x7fffffff (two 31-bit rand() results of
 * DQN::selectAction, src/dqn.cpp:30-33). */
uint64_t xq_rng(uint64_t seed, uint64_t env_id, uint32_t ctr);
/* smallest T such that (double)c/RAND_MAX < eps <=> c < T (src/dqn.cpp:30-31) */
uint32_t xq_eps_threshold(double eps);

/* ---- batched environment: replaces one ChessBoard + the board-facing half of ChessAI ---- */
/* n_envs boards on `device`, all at the standard opening (ChessBoard::ChessBoard/initializeBoard,
 * src/chessboard.cpp:4-29).  env_id0 = global id of env 0 (multi-GPU sharding keeps results
 * independent of the GPU count). */
int xq_env_create(int64_t n_envs, int device, uint64_t seed, uint64_t env_id0, xq_env_t* out);
int xq_env_destroy(xq_env_t h);
int xq_env_count(xq_env_t h, int64_t* n_envs);
int xq_env_set_stream(xq_env_t h, void* cuda_stream);
int xq_env_sync(xq_env_t h);
/* device address of the xq_env_rec array (for zero-copy consumers, e.g. the Q-network) */
int xq_env_device_boards(xq_env_t h, void** dev_ptr);
/* ChessBoard::reset, src/chessboard.cpp:95-102; mask_host[n] != 0 selects, NULL = all */
int xq_env_reset(xq_env_t h, const uint8_t* mask_host);
int xq_env_set_boards(xq_env_t h, const xq_env_rec* recs_host, int64_t first, int64_t n);
int xq_env_get_boards(xq_env_t h, xq_env_rec* recs_host, int64_t first, int64_t n);
/* ChessAI::getAllValidActions(currentPlayer) for every env, src/chessai.cpp:347-368 over
 * ChessBoard::getValidMoves + generate*Moves, src/chessboard.cpp:112-283, in reference order.
 * counts_host[n]; actions_host[n][XQ_MAX_ACTIONS], entries past the count are XQ_ACTION_NONE. */
int xq_env_legal_moves(xq_env_t h, uint8_t* counts_host, xq_action* actions_host);
/* OPT-IN, not a rule of the reference (which plays "capture the General": no king-safety test, no flying-general rule, SURVEY F1/F2;
 * every other entry point follows it bit-exactly): the list of xq_env_legal_moves, same order and layout, without the actions that
 * standard Xiangqi forbids -- after the action (a) some enemy piece would have the mover's General among the destinations
 * ChessBoard::getValidMoves generates for it (self-check), or (b) the two Generals would face each other on a file with nothing
 * between them (flying general).  "General" = the side's first General in square order; a side without one keeps every action. */
int xq_env_legal_moves_strict(xq_env_t h, uint8_t* counts_host, xq_action* actions_host);
/* ChessBoard::getValidMoves(row,col) for one square of every env (any colour), same order.
 * to_host[n][20], counts_host[n]. */
int xq_env_valid_moves(xq_env_t h, int row, int col, uint8_t* counts_host, uint8_t* to_host);
/* ChessBoard::isValidMove, src/chessboard.cpp:66-93 (+ :328-440): one query per env,
 * rows/cols may be off-board (=> 0).  moves_host[n][4] = fr,fc,tr,tc. */
int xq_env_is_valid_move(xq_env_t h, const int32_t* moves_host, uint8_t* valid_host);
/* ChessBoard::movePiece (src/chessboard.cpp:38-64) + ChessAI::evaluateBoard for the mover with
 * the post-move moveCount (src/chessai.cpp:115-116,311-345) + checkGameOver (:286-309) +
 * getWinner (:312-320).  A rejected action changes nothing (valid=0, captured=0).
 * auto_reset != 0: terminal envs are reset after their outputs are taken (chessai.cpp:90).
 * Any output pointer may be NULL. */
int xq_env_step(xq_env_t h, const xq_action* actions_host, int32_t* reward_host, uint8_t* done_host,
                uint8_t* winner_host, uint8_t* captured_host, uint8_t* valid_host, int auto_reset);
/* API mode without host traffic (a caller whose policy also lives on the device): the same three steps, asynchronous on the handle's stream,
 * results in device buffers owned by the handle (valid until the next call of the same kind; any output pointer may be NULL).
 * xq_env_legal_moves_device: counts u8 [n], actions xq_action [n][XQ_MAX_ACTIONS] (xq_env_legal_moves).
 * xq_env_pick_random_device: the random policy of xq_env_rollout_random on the lists of the last xq_env_legal_moves_device call:
 *   action = list[idx31 % count] with idx31 from xq_rng(seed, env id, the env's ply counter) (XQ_ACTION_NONE for an empty list) -> xq_action [n].
 * xq_env_step_device: xq_env_step on device actions (NULL = the actions xq_env_pick_random_device chose); reward i32 [n], the rest u8 [n]. */
int xq_env_legal_moves_device(xq_env_t h, void** counts_dev, void** actions_dev);
int xq_env_pick_random_device(xq_env_t h, void** actions_dev);
int xq_env_step_device(xq_env_t h, const void* actions_dev, int auto_reset, void** reward_dev, void** done_dev, void** winner_dev,
                       void** captured_dev, void** valid_dev);
/* Fused random-policy self-play: n_plies iterations of the ChessAI::train loop body without the
 * network (src/chessai.cpp:96-119): ordered list -> list[idx31 % n] -> movePiece -> evaluateBoard
 * -> checkGameOver, reset on terminal.  One launch; boards stay on chip between plies.
 * trace_host[n_plies][n_envs] and stats_host may be NULL. */
int xq_env_rollout_random(xq_env_t h, int n_plies, xq_trace_rec* trace_host, xq_env_stats* stats_host);
/* Host boards in, host boards out, ONE call: xq_env_set_boards(boards_in) + xq_env_rollout_random + xq_env_get_boards(boards_out)
 * enqueued back to back on the handle's stream with a single synchronisation at the end (three calls = three).  All n_envs boards;
 * boards_in_host may be NULL (continue from the boards on the device), as may boards_out_host, trace_host and stats_host. */
int xq_env_rollout_random_io(xq_env_t h, const xq_env_rec* boards_in_host, int n_plies, xq_env_rec* boards_out_host,
                             xq_trace_rec* trace_host, xq_env_stats* stats_host);
/* The same call in two halves, for a double-buffered caller (two env handles on one stream: the host submits the step of handle B before
 * it waits for the step of handle A, so launch latency and the host's wake-up hide under the other handle's kernel; the kernels of one
 * stream never overlap).  _submit enqueues [boards in -> rollout -> boards / trace / stats out] and returns; _wait blocks until that
 * step's outputs are in host memory.  The copies run on copy streams owned by the handle, ordered against the rollout by events: the boards
 * of the next step arrive and the results of the previous step leave while the other handle's kernel runs.  The host buffers and the handle
 * belong to the library between the two calls: one submission per handle at a time, every other call on the handle is refused until _wait
 * (XQ_ERR_STATE).  Results are identical to xq_env_rollout_random_io (which reads / writes pinned buffers from inside the kernel instead). */
int xq_env_rollout_random_io_submit(xq_env_t h, const xq_env_rec* boards_in_host, int n_plies, xq_env_rec* boards_out_host,
                                    xq_trace_rec* trace_host, xq_env_stats* stats_host);
int xq_env_rollout_random_io_wait(xq_env_t h);
/* same, device-resident and asynchronous: no host traffic; stats accumulate on the device */
int xq_env_rollout_random_async(xq_env_t h, int n_plies);
/* same with the per-ply trace [n_plies][n_envs] written to a device buffer owned by the handle (*trace_dev, valid until the next traced
 * call; may be NULL): the traced mode without host traffic */
int xq_env_rollout_random_traced_async(xq_env_t h, int n_plies, void** trace_dev);
int xq_env_get_stats(xq_env_t h, xq_env_stats* stats_host, int reset);
/* ChessAI::getStateRepresentation, src/chessai.cpp:268-289: out_host[n][1260] doubles */
int xq_env_state_onehot(xq_env_t h, double* out_host);

/* ---- device-resident interface for a policy that is not the library's DQN (a CNN, an actor-critic, ...) ----
 * All three calls are asynchronous on the handle's stream and write into CALLER-PROVIDED device buffers (a torch tensor's data_ptr()
 * can be passed straight in); the handle keeps no outputs.  Any optional pointer may be NULL.  Same rules as every other entry point
 * (the reference's, not standard Xiangqi).
 *
 * View.  XQ_VIEW_ABSOLUTE is the reference's frame.  XQ_VIEW_SIDE_TO_MOVE shows an env with Black to move rotated by 180 degrees:
 * square s <-> 89 - s = (9-r)*9 + (8-c), and colours swapped (channels 0..6 the mover's pieces, 7..13 the opponent's).  The same
 * mapping applies to observation planes, mask indices, score indices and given / returned actions.  Envs with Red to move (and envs
 * whose player byte is not 0 or 1) are not transformed.
 * Policy index.  from*90 + to in the frame of the view: XQ_POLICY_ACTIONS = 8,100 entries, the output width of the reference network. */
enum { XQ_DTYPE_F32 = 0, XQ_DTYPE_BF16 = 1, XQ_DTYPE_U8 = 2 };
enum { XQ_VIEW_ABSOLUTE = 0, XQ_VIEW_SIDE_TO_MOVE = 1 };
enum { XQ_PICK_GREEDY = 0, XQ_PICK_SAMPLE = 1, XQ_PICK_GIVEN = 2 };
#define XQ_POLICY_ACTIONS 8100            /* policy index = from*90 + to, in the frame of `view` */
#define XQ_MASK_WORDS 254                 /* packed mask: ceil(8100/32) uint32 per env, bits >= 8100 zero */

/* Observation: planes_dev[n][14][10][9] of 0/1 in f32, bf16 or u8 (dtype).  Absolute view: channel code-1 holds the reference's
 * one-hot, planes[e][ch][s] == getStateRepresentation[s*14 + ch] (src/chessai.cpp:268-289).  aux_dev[n][4] int32 = player, move_count,
 * red_score, black_score, always in absolute terms.  planes_dev must be 16-byte aligned. */
int xq_env_observe_device(xq_env_t h, void* planes_dev, int dtype, int view, int32_t* aux_dev);
/* Legal-action mask: the set of ChessAI::getAllValidActions(currentPlayer) (src/chessai.cpp:347-368) as policy indices.
 * packed != 0: uint32 [n][XQ_MASK_WORDS], index i is bit i%32 of word i/32 (for rollout buffers, 1 KB per env).
 * packed == 0: uint8 [n][8100] of 0/1 (usable as a torch.bool for masked_fill, 8 KB per env).  mask_dev must be 16-byte aligned. */
int xq_env_legal_mask_device(xq_env_t h, void* mask_dev, int packed, int view);
/* One ply for every env from a policy's output, one call: move generation, the choice, ChessBoard::movePiece, reward, terminal, winner
 * and the optional reset; the outputs after the choice are exactly those of xq_env_step_device with the chosen action.
 * scores_dev: [n][8100] f32 or bf16 (scores_dtype), contiguous, in the view's frame; only the entries of legal actions are read.
 * Cleaned scores: NaN counts as -inf, +inf as FLT_MAX.
 *  XQ_PICK_GREEDY: the FIRST legal action in reference list order with the largest score (strict >, as DQN::selectAction).
 *  XQ_PICK_SAMPLE: a draw from softmax(score / temperature) over the legal actions.  x = xq_rng(seed, env_id0 + e, rec.ctr),
 *    u = (float)(x >> 40) * 2^-24; m = max, S = sum of exp((l_k - m) / T) in reference list order; the action is the first k whose
 *    running sum exceeds u*S (the last legal action if rounding leaves none).  The draw uses the env's ply counter: results do not
 *    depend on how envs are sharded over handles or GPUs.
 *  XQ_PICK_GIVEN: actions_dev (int64 policy indices, -1 = none) is read, not written.  An index outside [0, 8100) or not legal is
 *    rejected like an xq_env_step action: valid = 0, the board is unchanged.  With scores_dev non-NULL, logp is the given action's
 *    log-probability (PPO's re-evaluation of stored actions).
 * If every legal score is -inf (or NaN) the first action in reference order is played, and logp is NaN.  An empty list (also any env
 * whose player byte is not 0 or 1) behaves like xq_env_step_device with XQ_ACTION_NONE.
 * Outputs: actions_dev (GREEDY / SAMPLE) int64 [n] = the chosen policy index, -1 for an empty list; logp_dev f32 [n] = (l_k - m)/T - log S
 * of the played action (NaN when not defined: empty list, rejected or scoreless GIVEN); reward i32 [n]; done, winner, captured, valid u8 [n].
 * temperature must be finite and > 0 for SAMPLE and whenever logp is computed; otherwise the call returns XQ_ERR_INVALID. */
int xq_env_policy_step_device(xq_env_t h, const void* scores_dev, int scores_dtype, int pick, float temperature, int view,
                              int auto_reset, int64_t* actions_dev, float* logp_dev, int32_t* reward_dev, uint8_t* done_dev,
                              uint8_t* winner_dev, uint8_t* captured_dev, uint8_t* valid_dev);

/* ---- device-resident batched tree search (PUCT / MCTS) for an external policy/value network ----
 * One tree per env of an env handle; each simulation selects one leaf per tree, the caller evaluates all leaves with ONE network call
 * and hands back scores and values; everything in between stays on the device.  Every call is asynchronous on the env handle's stream
 * and device; destroy the search before the env.  Same rules as every other entry point (the reference's).
 *
 * Tree.  The root is the env's record at xq_search_reset.  A node holds its board as an xq_env_rec; a child's record equals, bit for bit,
 * what xq_env_step_device (auto_reset = 0) makes of the parent's record and the edge's action (move_count, player, scores, ctr included).
 * Edges are a node's legal actions in reference list order (xq_env_legal_moves; the first 128), each with the prior P, the visit count N,
 * the value sum W (from the side to move at the parent) and the child.  N_node = simulations whose path contained the node, leaf included.
 * Selection (one leaf per tree per simulation, no virtual loss), from the root: a node not yet expanded, or terminal, is the leaf;
 * otherwise the edge with the largest Q + U, ties to the smaller list index, in f32 with no contraction, in this order:
 *   Q = N > 0 ? W / N : fpu,   U = ((c_puct * P) * sqrt(N_node)) / (1 + N).
 * If that edge has no child yet, the child is made and is the leaf: a simulation adds at most one node per tree.
 * Leaf status (u8): 0 needs evaluation, 1 a General was captured, 2 move cap (move_count >= 200), 3 no legal action (known once the node
 * was expanded to zero edges: the first simulation that reaches such a node reports 0, later ones 3).  A General captured on the 200th
 * ply is status 1.  Also per tree: winner (as xq_env_step: getWinner), the reward of the move that made the leaf (0 at the root), the
 * depth (plies below the root).
 * Expansion (status 0 only): scores [n][8100] (f32 / bf16, in the frame of `view`, cleaned as in xq_env_policy_step_device; only legal
 * entries are read) give P_k = exp((l_k - m) / T) / S, S summed in list order, uniform 1 / count if every legal score is -inf.  At the root
 * only, with root_noise_dev [n][8100] f32 (finite; e.g. Dirichlet noise the caller draws over the legal mask):
 * P <- (1 - eps) * P + eps * noise[index].  The library draws no random numbers.
 * Backup (every status): the caller's value of the leaf, from the leaf's side to move, NaN -> 0, clamped to [-1, 1]; going up,
 * v <- -v, the edge gets N += 1 and W += v, every node on the path N_node += 1.  The library has no value convention for terminal leaves.
 *
 * Call order: xq_search_reset, then per simulation select -> (leaves / observe_leaves, any number of times) -> expand_backup; anything
 * else is XQ_ERR_STATE, as is a select past max_simulations since the reset.  root_device and get_tree work at any time after a reset.
 * Memory: (max_simulations + 1) x 2,389 + 73 bytes per tree (xq_search_bytes_per_tree): per node a record, 21 bytes of node state and
 * 128 edge slots of 18 bytes (P, N, W, child, action); per tree the leaf record and 9 bytes. */
typedef struct xq_search_s* xq_search_t;
#define XQ_SEARCH_MAX_EDGES 128
typedef struct {
    xq_env_rec rec;       /* the node's board */
    int32_t parent;       /* node index in the tree, -1 at the root (node 0) */
    int32_t visits;       /* N_node */
    int32_t reward;       /* reward of the move that made the node (0 at the root) */
    int32_t depth;        /* plies below the root */
    uint8_t parent_edge;  /* list index of the edge from the parent */
    uint8_t n_edges;      /* edges after expansion */
    uint8_t expanded;
    uint8_t status;       /* 0 not terminal, 1 General captured, 2 move cap, 3 expanded without a legal action */
    uint8_t winner;       /* getWinner of the node's board */
    uint8_t reserved[3];
} xq_search_node;         /* 88 B */
typedef struct {
    int32_t action;       /* absolute policy index from * 90 + to, -1 past n_edges */
    float prior;
    int32_t visits;       /* N */
    float value_sum;      /* W, from the side to move at the parent */
    int32_t child;        /* node index, -1 none */
} xq_search_edge;         /* 20 B */

/* capacity max_simulations + 1 nodes per tree; XQ_ERR_NOMEM when the device memory cannot be had.  The trees are empty until a reset. */
int xq_search_create(xq_env_t env, int max_simulations, xq_search_t* out);
int xq_search_destroy(xq_search_t s);
int xq_search_bytes_per_tree(int max_simulations, int64_t* bytes);
/* roots = the env's current records (read in stream order), every tree empty, simulation count 0 */
int xq_search_reset(xq_search_t s);
/* one leaf per tree; c_puct finite and >= 0, fpu finite.  Outputs [n] (any may be NULL): status u8, winner u8, reward i32, depth i32 */
int xq_search_select_device(xq_search_t s, float c_puct, float fpu, uint8_t* status_dev, uint8_t* winner_dev, int32_t* reward_dev,
                            int32_t* depth_dev);
/* device address of the [n] leaf records of the last selection (valid until the next select) */
int xq_search_leaves_device(xq_search_t s, void** leaf_recs_dev);
/* xq_env_observe_device on the leaf records: same planes / aux contract */
int xq_search_observe_leaves_device(xq_search_t s, void* planes_dev, int dtype, int view, int32_t* aux_dev);
/* expansion of the status-0 leaves and backup of every leaf: scores_dev [n][8100] (scores_dtype f32 / bf16), temperature finite > 0,
 * values_dev f32 [n] (required), root_noise_dev f32 [n][8100] or NULL, noise_eps in [0, 1] */
int xq_search_expand_backup_device(xq_search_t s, const void* scores_dev, int scores_dtype, float temperature, int view,
                                   const float* values_dev, const float* root_noise_dev, float noise_eps);
/* per root (any output may be NULL): visits_dev int32 [n][8100] (16-byte aligned) = the root edges' N at their policy indices in the frame
 * of `view`, 0 elsewhere; q_dev f32 [n] = sum W / sum N over the root's edges (sums in list order; NaN when no edge was visited); best_dev
 * int64 [n] = policy index (frame of `view`) of the most-visited root edge, first in list order on ties, -1 when no edge was visited --
 * the input of xq_env_policy_step_device with XQ_PICK_GIVEN. */
int xq_search_root_device(xq_search_t s, int view, int32_t* visits_dev, float* q_dev, int64_t* best_dev);
/* synchronous read-back of one tree: nodes_host[max_simulations + 1], edges_host [max_simulations + 1][128] (may be NULL; edges past a
 * node's n_edges have action -1 and child -1), *n_nodes = nodes in the tree */
int xq_search_get_tree(xq_search_t s, int64_t tree, xq_search_node* nodes_host, xq_search_edge* edges_host, int32_t* n_nodes);

/* ---- DQN: replaces DQN (include/dqn.h:97-116, src/dqn.cpp) + NeuralNetwork (include/dqn.h:43-95, src/dqn.cu) ----
 * Parameters use the reference layout (src/dqn.cu:112-140): weights = layer after layer, each [out][in]
 * row-major; biases = layer after layer.
 * Two numeric paths:
 *  (1) FP64, any layer sizes, per-sample semantics identical to the reference's kernels: xq_dqn_forward,
 *      xq_dqn_backprop, xq_dqn_select_action, xq_dqn_train.  Tolerance vs the reference: 1e-12 abs
 *      (summation order and FMA contraction differ in the last ulps).
 *  (2) batched BF16 tensor-core path for the {1260,128,8100} self-play network, fed by packed boards:
 *      xq_dqn_forward_boards, xq_dqn_act, xq_dqn_td_update.  FP32 master weights, BF16 MMA operands, FP32
 *      accumulation.  Tolerance vs the FP64 oracle: |dQ| <= 2e-3 abs. */
typedef struct xq_dqn_s* xq_dqn_t;
enum { XQ_DQN_AS_WRITTEN = 0, XQ_DQN_CORRECTED = 1 };   /* hidden-layer delta: src/dqn.cu:406-427 as written, or W^T.delta (SURVEY F7) */

/* NeuralNetwork::NeuralNetwork + initializeHostWeightsAndBiases (src/dqn.cu:14-57,96-146): W ~ U(-0.05,0.05) from
 * mt19937(seed) (the reference seeds from random_device), b = 0; DQN::DQN (src/dqn.cpp:12-20) copies it to the target. */
int xq_dqn_create(const int32_t* layer_sizes, int n_layers, double lr, double gamma, int device, uint64_t seed, int mode,
                  xq_dqn_t* out);
int xq_dqn_destroy(xq_dqn_t h);
int xq_dqn_set_stream(xq_dqn_t h, void* cuda_stream);
int xq_dqn_sync(xq_dqn_t h);
int xq_dqn_num_params(xq_dqn_t h, int64_t* n_weights, int64_t* n_biases);
/* host_weights / host_biases + copyToDevice (src/dqn.cu:480-485); also refreshes the target network like DQN::DQN */
int xq_dqn_set_params(xq_dqn_t h, const double* weights_host, const double* biases_host);
/* copyFromDevice (src/dqn.cu:487-492): the TRAINED parameters (the reference never calls it, SURVEY F10) */
int xq_dqn_get_params(xq_dqn_t h, double* weights_host, double* biases_host);
/* DQN::getQValues -> NeuralNetwork::forward (src/dqn.cpp:65-68, src/dqn.cu:184-260) for n states: q_host[n][out] */
int xq_dqn_forward(xq_dqn_t h, const double* states_host, int64_t n, double* q_host);
/* DQN::backpropagate -> NeuralNetwork::backpropagate (src/dqn.cpp:59-62, src/dqn.cu:275-467): n SEQUENTIAL SGD steps */
int xq_dqn_backprop(xq_dqn_t h, const double* states_host, const double* targets_host, int64_t n, double lr);
/* DQN::selectAction (src/dqn.cpp:24-56) with its two rand() results supplied (coin31, idx31); *index_out = list index */
int xq_dqn_select_action(xq_dqn_t h, const double* state_host, double eps, const xq_action* actions_host, int n_actions,
                         uint32_t coin31, uint32_t idx31, int* index_out);
/* one TD step on (s, a, r, s', done): target = Q(s); target[a] = done ? r : r + gamma * max Q'(s'); backprop(s, target).
 * use_target_net = 0: bootstrap from the online net = the live loop ChessAI::train (src/chessai.cpp:121-131);
 * use_target_net = 1: DQN::train (src/dqn.cpp:157-172).  lr <= 0 uses the handle's learning rate. */
int xq_dqn_train(xq_dqn_t h, const double* state_host, int action_index, double reward, const double* next_state_host,
                 int done, int use_target_net, double lr);
/* DQN::updateTargetNetwork (src/dqn.cpp:71-73); copies the live device weights (the evident intent, SURVEY F10) */
int xq_dqn_sync_target(xq_dqn_t h);
/* DQN::saveModel / loadModel byte layout (src/dqn.cpp:76-154): raw f64 weights | raw f64 biases | BE u64 n | n x BE i32 */
int xq_dqn_save(xq_dqn_t h, const char* path);
int xq_dqn_load(xq_dqn_t h, const char* path);

/* ---- batched tensor-core path ({1260,128,8100} only) ---- */
/* One replay transition, 128 B: packed board before (s) and after (s2) the move, the action, the mover's
 * colour, done and ChessAI::evaluateBoard's reward (src/chessai.cpp:113-119).  `done` follows the caller's
 * loop: checkGameOver() (startSelfPlay :227) or checkGameOver() || moveCount+1 >= 200 (train :119). */
typedef struct {
    uint32_t s[12];
    uint32_t s2[12];
    xq_action action;
    uint8_t mover;
    uint8_t done;
    int32_t reward;
    uint32_t reserved[6];
} xq_transition;

/* Q(s) for n packed boards through the tensor-core path: q_host[n][8100] FP32 (parity / debugging;
 * the training kernels never materialise Q) */
int xq_dqn_forward_boards(xq_dqn_t h, const xq_env_rec* boards_host, int64_t n, float* q_host);
/* One batched TD update (the body of ChessAI::train, src/chessai.cpp:121-131, for n transitions at once):
 * target_b = done ? r : r + gamma * max_a Q'(s2_b)[a]; loss 1/2 (Q(s_b)[to_b] - target_b)^2; gradients of all
 * samples are taken at the same weights and SUMMED, then W -= lr * grad (n = 1 is one reference step).
 * use_target_net: Q' = target network (DQN::train, src/dqn.cpp:157-172) instead of the online one.
 * lr <= 0 uses the handle's rate.  info_host[4] = {sum of losses, sum Q(s)[to], sum target, 0}. */
int xq_dqn_td_update(xq_dqn_t h, const xq_transition* batch_host, int64_t n, int use_target_net, double lr, float* info_host);
/* same on a device-resident batch, asynchronous; apply = 0 only accumulates the gradient (multi-GPU:
 * all-reduce xq_dqn_grad_buffer across ranks, then xq_dqn_apply_grads on every rank) */
int xq_dqn_td_update_device(xq_dqn_t h, const void* batch_dev, int64_t n, int use_target_net, double lr, int apply);
/* compact gradient of a TD step: [dW0^T 1260x128 | db0 128 | dW1 rows 0..89 x128 | db1 0..89] = 173,018 FP32 */
int xq_dqn_grad_buffer(xq_dqn_t h, void** dev_ptr, int64_t* n_floats);
int xq_dqn_apply_grads(xq_dqn_t h, double lr);

/* ---- multi-GPU: the one exchange step of the path (SURVEY 8e), fused with the SGD step, over peer memory ----
 * One process per GPU.  xq_dqn_dist_export returns the 64-byte CUDA IPC handle of this rank's gradient exchange buffer; the
 * ranks gather each other's handles with whatever transport they have (torch.distributed, MPI, a file) and pass all `world`
 * of them, in rank order, to xq_dqn_dist_connect.  From then on xq_dqn_td_update_*(apply = 0) leaves the compact gradient in
 * the exchange buffer and xq_dqn_dist_allreduce_apply launches ONE kernel per rank that signals / waits through flags in
 * peer memory, sums the world gradients in rank order over NVLink (bit-identical on every rank) and applies W -= lr * sum.
 * It replaces ncclAllReduce + xq_dqn_apply_grads.
 * EVERY applied update on a connected handle exchanges its gradient: xq_dqn_td_update / xq_dqn_td_update_device / _replay with apply = 1 and
 * xq_dqn_td_update_replay_n run the exchange INSIDE the gradient contraction kernel (contraction -> reduce-scatter of the 16-row blocks to
 * their owner ranks -> all-gather of the sums -> SGD, flag-in-data lines over peer memory).  Every rank must make the same sequence of update calls.
 * A wait for a peer that lasts longer than XQ_DIST_TIMEOUT_MS (default 20000) does NOT apply the update and makes the handle fail
 * (XQ_ERR_STATE, sticky) on every later update / exchange call: the replicas may differ, recreate the handles.
 * xq_dqn_dist_status: timed_out = epoch of the first exchange that timed out (0 = none).
 * xq_dqn_dist_info: rank / world of a connected handle (0 / 1 otherwise).
 * xq_dqn_dist_allgather: host-level all-gather of one message of `bytes` (<= 65536) per rank through the same peer-mapped buffer
 * (recv_host[world][bytes], rank order); collective and synchronous -- what xq_train_run uses to merge the ranks' finished games. */
#define XQ_IPC_HANDLE_BYTES 64
int xq_dqn_dist_export(xq_dqn_t h, void* handle_out);
int xq_dqn_dist_connect(xq_dqn_t h, int rank, int world, const void* handles);
int xq_dqn_dist_allreduce_apply(xq_dqn_t h, double lr);
int xq_dqn_dist_status(xq_dqn_t h, int* timed_out);
int xq_dqn_dist_info(xq_dqn_t h, int* rank, int* world);
int xq_dqn_dist_allgather(xq_dqn_t h, const void* send_host, int64_t bytes, void* recv_host);

/* ---- GPU-resident replay buffer + epsilon-greedy self-play (new capabilities: the reference trains online at
 * batch 1 and has no replay buffer, SURVEY F10; semantics are per transition those of ChessAI::train) ---- */
typedef struct xq_replay_s* xq_replay_t;
/* ring of `capacity` xq_transition records (128 B each: 1M transitions = 128 MB of HBM) */
int xq_replay_create(int64_t capacity, int device, xq_replay_t* out);
int xq_replay_destroy(xq_replay_t r);
int xq_replay_info(xq_replay_t r, int64_t* size, int64_t* capacity, int64_t* total_inserted);
/* batched insert of n host transitions at the ring head */
int xq_replay_insert(xq_replay_t r, const xq_transition* batch_host, int64_t n);
/* raw ring slots [first, first+n) (tests / checkpointing) */
int xq_replay_get(xq_replay_t r, int64_t first, int64_t n, xq_transition* out_host);
/* uniform sampling with replacement: index_i = (xq_rng(seed, i, counter) >> 1) % size.  Either output may be NULL. */
int xq_replay_sample(xq_replay_t r, int64_t batch, uint64_t seed, uint32_t counter, xq_transition* out_host, int64_t* index_host);

/* DQN::selectAction for every env at once (src/dqn.cpp:24-56 over ChessAI::getAllValidActions): coin31/idx31 come from
 * xq_rng(seed, env_id, ctr); explore: list[idx31 % n]; exploit: FIRST action maximising Q(s)[action.to] (strict >).
 * Nothing is applied.  q_host (optional) [n][96]: Q(s)[0..89] as used for the choice. */
int xq_dqn_act(xq_dqn_t h, xq_env_t env, double eps, xq_action* actions_host, float* q_host);
/* n_plies of epsilon-greedy self-play on every env, device-resident and asynchronous: per ply the body of ChessAI::train
 * (src/chessai.cpp:96-119) up to the transition (s, a, r, s', done), which is written to the replay ring (r may be NULL);
 * terminal envs restart.  train_done != 0: done = checkGameOver() || moveCount+1 >= 200 (train, :119), else checkGameOver()
 * (startSelfPlay, :227).  Env statistics accumulate in the env handle (xq_env_get_stats). */
int xq_selfplay_collect(xq_dqn_t h, xq_env_t env, xq_replay_t r, int n_plies, double eps, int train_done);
/* sample `batch` transitions from the ring and run xq_dqn_td_update_device on them, all on the device */
int xq_dqn_td_update_replay(xq_dqn_t h, xq_replay_t r, int64_t batch, uint64_t seed, uint32_t counter, int use_target_net, double lr,
                            int apply);

/* n_updates consecutive updates, counters counter0, counter0 + 1, ...: the same result, bit for bit, as n_updates calls of
 * xq_dqn_td_update_replay(..., apply = 1).  With use_target_net != 0 the updates are software-pipelined: the bootstrap branch
 * (h(s') with the target net + the [batch x 128] x [128 x 8100] row-max GEMM) of the next updates does not depend on the online
 * weights and runs on a second stream underneath the online branch of the current one.  On a handle connected to its peers
 * (xq_dqn_dist_connect) every update exchanges its gradient inside its contraction kernel. */
int xq_dqn_td_update_replay_n(xq_dqn_t h, xq_replay_t r, int64_t batch, uint64_t seed, uint32_t counter0, int n_updates, int use_target_net,
                              double lr);

/* ---- episode driver: the batched equivalent of ChessAI::train / startSelfPlay (src/chessai.cpp:85-170, :191-266) ----
 * One finished game of the self-play collector = the arguments of the reference's gameCompleted(game, redScore, blackScore)
 * signal (src/chessai.cpp:161) plus what its log line and statistics need. */
typedef struct {
    uint32_t ply;          /* collector ply (counted since xq_env_enable_game_events) at which the game ended */
    uint32_t env;          /* env index within this handle */
    int32_t red_score;     /* ChessBoard::getRedScore / getBlackScore when the game ended */
    int32_t black_score;
    uint16_t moves;        /* ChessBoard::getMoveCount */
    uint8_t winner;        /* ChessBoard::getWinner: 0 Red, 1 Black, 2 None */
    uint8_t reason;        /* 0 a General was captured, 1 move cap (200), 2 no legal action (:100-103) */
    uint32_t reserved;
} xq_game_event;           /* 24 B */
/* device ring of `capacity` finished-game events filled by xq_selfplay_collect; xq_env_drain_game_events copies the pending
 * events out SORTED by (ply, env) -- the deterministic game order of the batched loop -- and empties the ring;
 * *n_dropped = events lost because the ring was full since the last drain */
int xq_env_enable_game_events(xq_env_t h, int64_t capacity);
int xq_env_drain_game_events(xq_env_t h, xq_game_event* out_host, int64_t max_events, int64_t* n_out, int64_t* n_dropped);

typedef void (*xq_game_completed_fn)(void* user, int64_t game_number, int32_t red_score, int32_t black_score);
typedef struct {
    int64_t n_games;           /* stop after this many finished games (numEpisodes / numGames) */
    int plies_per_round;       /* self-play plies collected between two learning phases */
    int updates_per_round;     /* TD updates (batch `batch`) per learning phase; 0 = self-play only (startSelfPlay without training) */
    int64_t batch;
    double eps;                /* 0.1 in the reference (:106, :210) */
    double lr;                 /* <= 0: the network's rate (0.001, include/chessai.h:48) */
    int use_target_net;        /* 1: DQN::train bootstrap (src/dqn.cpp:157-172); 0: online net (ChessAI::train, :119-128) */
    int target_sync_plies;     /* updateTargetNetwork cadence in collector plies (the reference: every 100 plies, :140) */
    int train_done;            /* 1: done also when moveCount + 1 >= 200 (train, :119); 0: checkGameOver only (startSelfPlay, :227) */
    int autosave_games;        /* saveModel every this many games (100 in the reference, :165-167); 0 = never */
    const char* autosave_prefix;   /* file = "<prefix><games>_games.bin" ("model_after_" in the reference); NULL = that default */
    const char* log_path;      /* game_log.txt sink in ChessAI::onGameCompleted's line format (:370-393); NULL = none */
    uint64_t sample_seed;      /* replay sampling seed (xq_replay_sample) */
} xq_train_config;
typedef struct {
    int64_t games, plies, transitions, updates, target_syncs, autosaves, events_dropped;
    int64_t red_wins, black_wins;      /* by score, as the log line decides ("Red wins!" / "Black wins!" / "It's a draw!") */
    double seconds;
} xq_train_report;
/* Runs rounds of [collect plies_per_round plies over all envs -> updates_per_round TD updates -> drain the finished games in
 * (ply, env) order: callback (gameCompleted), log line, autosave] until n_games games have finished.  Synchronous.
 * autosave: one snapshot per round in which a multiple of autosave_games was crossed, named after the last crossed multiple (the
 * weights at the end of that round).
 * Multi-GPU = BASELINE config 4 as ONE call per rank: when `h` is connected to its peers (xq_dqn_dist_connect) every rank calls this
 * with its own env / replay shard and the same cfg; n_games, the game numbers, the report's games / transitions / wins count the games
 * of ALL ranks merged in (ply, global env) order (identical on every rank and for every GPU count of the same total env range); the
 * callback fires on every rank that passes one, the log file and the autosaves are written by rank 0 only. */
int xq_train_run(xq_dqn_t h, xq_env_t env, xq_replay_t r, const xq_train_config* cfg, xq_game_completed_fn cb, void* user, xq_train_report* report);

/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
uint64_t xq_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif
