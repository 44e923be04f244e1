/* bgx.h — C-ABI of libbgx, the B200-native batched backgammon self-play engine.
 *
 * This is the drop-in boundary for ONE hot path of romanoshiliarhopoulos/Backgammon-Engine:
 *   enumerate every legal afterstate of (position, dice)  ->  encode 198 features  ->
 *   score with the 198-128-1 sigmoid MLP  ->  argmax/argmin  ->  apply  ->  TD(lambda) update.
 * The reference binds that path to Python through cppsrc/backgammon_bindings.cpp; the
 * entry points below are what that binding file would call instead (INTEGRATION.md shows
 * the pybind11 stubs).  Plain C types only: pointers + sizes, caller-allocated buffers,
 * no exceptions; every function returns 0 on success or a negative BGX_E_* code and
 * leaves a message in bgx_last_error() (thread-local).
 *
 * Citations "file:line" are relative to the reference checkout.
 *
 * POSITION  = the reference's TurnEval row (cppsrc/game.hpp:17-28), 28 ints:
 *             [0..23] board (+ PLAYER1 / - PLAYER2, index = point-1),
 *             [24] jailed P1, [25] jailed P2, [26] borne-off P1, [27] borne-off P2.
 * RECORD    = the 32-byte int8 form every batched call uses:
 *             bytes 0..27 the position, byte 28 player to move (0/1), byte 29 die 1,
 *             byte 30 die 2, byte 31 reserved (0).  Arrays of records are 32-byte strided,
 *             so one warp reads/writes a record as one 32-byte sector.
 * MOVES     = a turn sequence: up to 4 (origin, dest) int8 pairs, origin/dest coded as the
 *             reference does (0 = P1 bar / P2 off, 1..24 points, 25 = P2 bar / P1 off).
 * WEIGHTS   = the reference state_dict tensors (model.py:36-37), fp32, row-major:
 *             W1[128][198] fc1.weight, b1[128] fc1.bias, w2[128] fc2.weight, b2[1] fc2.bias.
 *
 * The batched entry points run on the GPU only.  There is no CPU fallback: without a
 * CUDA device bgx_create fails with BGX_E_NO_DEVICE and nothing batched can be called.
 * The single-position functions (section 1) are host code; they back the per-object
 * compat API (Game.legalMoves, Game.tryMove ...) whose cost is Python-call bound.
 */
#ifndef BGX_H
#define BGX_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BGX_STATE_INTS 28
#define BGX_RECORD_BYTES 32
#define BGX_FEATURES 198
#define BGX_HIDDEN 128
#define BGX_NPARAMS 25601          /* 198*128 + 128 + 128 + 1 */
#define BGX_NPARAMS_PADDED 25604   /* 16-byte multiple: the allreduce message */

enum {
    BGX_OK = 0,
    BGX_E_INVALID = -1,      /* bad argument */
    BGX_E_NO_DEVICE = -2,    /* no CUDA device / driver: the batched path cannot run */
    BGX_E_CUDA = -3,         /* a CUDA call failed; see bgx_last_error() */
    BGX_E_CAPACITY = -4,     /* caller buffer too small; *needed is filled */
    BGX_E_STATE = -5         /* call order (e.g. selfplay step before init, weights unset) */
};

/* tryMove outcome codes; bgx_move_error_string() gives the reference's exact text
 * (cppsrc/game.cpp:585-642). */
enum {
    BGX_MOVE_OK = 0,
    BGX_MOVE_INVALID_ORIGIN = 1,
    BGX_MOVE_ORIGIN_RANGE = 2,
    BGX_MOVE_DEST_RANGE = 3,
    BGX_MOVE_DIRECTION = 4,
    BGX_MOVE_DICE = 5,
    BGX_MOVE_INVALID_DEST = 6,
    BGX_MOVE_BEAR_FROM_JAIL = 7
};

const char *bgx_last_error(void);
int bgx_abi_version(void);

/* ------------------------------------------------------------------------------------
 * 1. Single-position host functions (compat Game object)
 * ---------------------------------------------------------------------------------- */

/* replaces Game::legalMoves(player, die)                      cppsrc/game.cpp:80-105
 * out_pairs[2*i], out_pairs[2*i+1] = origin, dest; at most 26 pairs. */
int bgx_legal_moves(const int32_t *position, int player, int die, int8_t *out_pairs, int cap, int *n);

/* replaces Game::tryMove(player*, dice, origin, dest, err)     cppsrc/game.cpp:573-663
 * position is updated in place on success; *move_code gets a BGX_MOVE_* value. */
int bgx_try_move(int32_t *position, int player, int dice, int origin, int dest, int *move_code);
const char *bgx_move_error_string(int move_code);

/* replaces Game::over(&winner) / is_game_over                  cppsrc/game.cpp:388-407,
 *                                                              backgammon_bindings.cpp:11-16
 * *winner = -1 while the game is running. */
int bgx_game_over(const int32_t *position, int *winner);

/* replaces Game::legalTurnSequences + Game::evaluateTurnSequences
 *                                                              cppsrc/game.cpp:134-222
 * seq_moves[cap][4][2], seq_len[cap], states[cap][28] (any may be NULL); reference order,
 * duplicates kept.  *n = number of sequences; BGX_E_CAPACITY if n > cap. */
int bgx_turn_sequences(const int32_t *position, int player, int d1, int d2, int64_t cap,
                       int8_t *seq_moves, int8_t *seq_len, int32_t *states, int64_t *n);

/* ------------------------------------------------------------------------------------
 * 2. Engine handle (one per device, not thread-safe)
 * ---------------------------------------------------------------------------------- */
typedef struct bgx_engine bgx_engine;

int bgx_device_count(int *n);
int bgx_create(int device, bgx_engine **out);
int bgx_destroy(bgx_engine *e);
/* all later launches of this engine go to `cuda_stream` (a cudaStream_t; NULL = default) */
int bgx_set_stream(bgx_engine *e, void *cuda_stream);
int bgx_synchronize(bgx_engine *e);

/* replaces model.load_state_dict / state_dict()               model.py:36-37, train.py:513-515
 * host pointers, WEIGHTS layout. */
int bgx_set_weights(bgx_engine *e, const float *W1, const float *b1, const float *w2, const float *b2);
/* (bgx_set_weights and bgx_apply_delta return BGX_E_STATE while an asynchronous lane holds a batch: its kernel reads the
 * weight tables on its own stream; bgx_lane_wait every busy lane first) */
int bgx_get_weights(bgx_engine *e, float *W1, float *b1, float *w2, float *b2);

/* ------------------------------------------------------------------------------------
 * 3. Batched position kernels.  `*_host` variants take HOST buffers and do the H2D/D2H
 *    copies themselves (the end-to-end path); the plain variants take DEVICE pointers
 *    and only enqueue work on the engine's stream.
 * ---------------------------------------------------------------------------------- */

/* Batched Game::evaluateTurnSequences, summary form            cppsrc/game.cpp:193-222
 * per query: number of sequences N (reference count, duplicates included), number of
 * distinct afterstates U (-1 if the exact-dedup table overflowed, never seen in practice),
 * and the order-dependent 64-bit digest over every (sequence, afterstate) — DESIGN.md
 * "enumeration digest" — that pins the ORDERED list bit-exactly without moving it. */
int bgx_enumerate_summary(bgx_engine *e, const int8_t *queries, int64_t n_queries,
                          int32_t *n_seq, int32_t *n_unique, uint64_t *digest);
int bgx_enumerate_summary_host(bgx_engine *e, const int8_t *queries, int64_t n_queries,
                               int32_t *n_seq, int32_t *n_unique, uint64_t *digest);

/* Batched Game::evaluateTurnSequences, materialised            cppsrc/game.cpp:193-222,
 *                                                              backgammon_bindings.cpp:27-39
 * offsets[n_queries+1] = exclusive prefix sum of N (from a previous summary call);
 * sequence k of query q lands at row offsets[q]+k: seq_moves[row][8], seq_len[row],
 * states[row][32] (RECORD, byte 28 = mover). */
int bgx_enumerate(bgx_engine *e, const int8_t *queries, int64_t n_queries, const int64_t *offsets,
                  int8_t *seq_moves, int8_t *seq_len, int8_t *states);
/* The allocation pass of the materialised form, on DEVICE buffers: n_seq[n] (int32) = size of every query's list
 * (a count-only walk: no distinct-afterstate table, no digest), offsets[n + 1] (int64) = their exclusive prefix sum,
 * offsets[n] = total rows.  What bgx_enumerate takes as `offsets`. */
int bgx_enumerate_count(bgx_engine *e, const int8_t *queries, int64_t n_queries, int32_t *n_seq, int64_t *offsets);
/* host convenience: count + device scan + enumerate; *total = sum N.  Output buffers hold
 * `cap` rows; BGX_E_CAPACITY (with *total set) when more are needed. offsets may be NULL. */
int bgx_enumerate_host(bgx_engine *e, const int8_t *queries, int64_t n_queries, int64_t cap,
                       int64_t *offsets, int8_t *seq_moves, int8_t *seq_len, int8_t *states,
                       int64_t *total);

/* replaces TDLGammonModel._encode_states_np(states, turn)      model.py:111-144
 * records[n][32] (byte 28 = the `turn` flag) -> X[n][198] fp32, bit-exact. */
int bgx_encode(bgx_engine *e, const int8_t *records, int64_t n, float *X);
int bgx_encode_host(bgx_engine *e, const int8_t *records, int64_t n, float *X);

/* replaces TDLGammonModel.forward(_encode_states_np(states, turn))   model.py:63-67
 * V[n] fp32; features are generated in-kernel, X never touches HBM. */
int bgx_evaluate(bgx_engine *e, const int8_t *records, int64_t n, float *V);
int bgx_evaluate_host(bgx_engine *e, const int8_t *records, int64_t n, float *V);

/* Batched TDLGammonModel.make_move(game, epsilon)              model.py:180-222
 * per query: enumerate, score every distinct afterstate with the mover's flag, take
 * argmax (P1) / argmin (P2) with the reference's first-index tie-break, or — with
 * probability epsilon — a uniformly random SEQUENCE (duplicates weighted like
 * random.randrange(len(actions)), model.py:205-206; draws come from Philox keyed by
 * (seed, query index)).  Outputs (any may be NULL):
 *   chosen[n][32]   afterstate RECORD; byte 28 = mover, byte 31 = 1 if a sequence was played
 *                   (0: no legal sequence, or the single empty sequence of a blocked double)
 *   moves[n][8], moves_len[n]   the chosen sequence
 *   value[n]        V of the chosen afterstate (NaN when nothing was scored)
 *   n_seq[n], n_scored[n]       sequences enumerated / afterstates actually scored */
int bgx_select_moves(bgx_engine *e, const int8_t *queries, int64_t n, float epsilon, uint64_t seed,
                     int8_t *chosen, int8_t *moves, int8_t *moves_len, float *value,
                     int32_t *n_seq, int32_t *n_scored);
int bgx_select_moves_host(bgx_engine *e, const int8_t *queries, int64_t n, float epsilon, uint64_t seed,
                          int8_t *chosen, int8_t *moves, int8_t *moves_len, float *value,
                          int32_t *n_seq, int32_t *n_scored);

/* Two-ply move selection: make_move's one-ply rule (model.py:180-222) looking one roll ahead.  Per query (s, mover p, dice):
 *   candidates   the distinct afterstates of the turn sequences, in order of first appearance in reference order, each with
 *                the first sequence that reaches it (n_candidates = U of bgx_enumerate_summary);
 *   a win        a candidate that bears off p's 15th checker is worth exactly 1 (PLAYER1) / 0 (PLAYER2); if there is one, the
 *                first such candidate is the pick and nothing is expanded;
 *   filter       max_candidates K = 0 expands every candidate; K > 0 the K best by one-ply value (the value bgx_select_moves
 *                compares, signed for p; first appearance on ties), so K = 1 picks what bgx_select_moves picks;
 *   expansion    for each of the opponent's 21 rolls (a = 1..6, b = 1..a, weight 2 if a != b) the reply value R is the value
 *                bgx_select_moves reports for (A, 1 - p, a, b); a blocked opponent (no sequence, or the empty one of a double)
 *                leaves V(A, 1 - p), bgx_evaluate's value; E2(A) = sum(weight * R) / 36 in float64, in that roll order, rounded once to fp32;
 *   pick         arg-max E2 (PLAYER1) / arg-min (PLAYER2), first appearance on ties.
 * Outputs (any may be NULL) mean what they mean for bgx_select_moves: chosen[n][32] (byte 28 = mover, byte 31 = 1 if a sequence
 * with a move was played), moves[n][8] / moves_len[n] the first sequence reaching the pick, value[n] its E2 (1 / 0 for a win,
 * NaN without a sequence), n_candidates[n], n_expanded[n].  A pure function of (query, weights, K).  The replies run through
 * bgx_select_moves' kernel in chunks of bgx_set_option "twoply_chunk" replies (0 = 2^21), so scratch stays bounded; the device
 * form synchronises the engine's stream twice to size its buffers.  BGX_E_CAPACITY if a query has more than 4096 distinct
 * afterstates (never seen: the largest U in 3,200 random games is 783). */
int bgx_select_moves_2ply(bgx_engine *e, const int8_t *queries, int64_t n, int32_t max_candidates,
                          int8_t *chosen, int8_t *moves, int8_t *moves_len, float *value,
                          int32_t *n_candidates, int32_t *n_expanded);
int bgx_select_moves_2ply_host(bgx_engine *e, const int8_t *queries, int64_t n, int32_t max_candidates,
                               int8_t *chosen, int8_t *moves, int8_t *moves_len, float *value,
                               int32_t *n_candidates, int32_t *n_expanded);

/* Rollouts: Monte Carlo evaluation of n positions (RECORDs: bytes 0..27 the position, byte 28 the player on roll, bytes 29..31
 * ignored) with bgx_select_moves' greedy one-ply policy (epsilon 0, make_move) on both sides.  Per position, `trials` independent
 * trials t = 0 .. trials-1, each played until the game ends or `max_plies` plies were played (0: to the end, with the hard cap
 * BGX_ROLLOUT_MAX_PLIES applied the same way):
 *   dice       ply k of trial t (k = 0: the player on roll) rolls Philox4x32-10, key = seed, counter = (k, t lo, t hi, 4), dice as
 *              self-play draws them; with BGX_ROLLOUT_STRATIFY ply 0 rolls r = t mod 36 instead (d1 = 1 + r / 6, d2 = 1 + r % 6), and
 *              trials must be a multiple of 36.  Dice depend on the trial index only: every position of a batch sees the same dice
 *              (common random numbers), and results do not depend on batching;
 *   a ply      is bgx_select_moves at epsilon 0; the game is over when byte 26 == 15 (PLAYER1 wins, checked first) or byte 27 == 15;
 *   x_t        a P(PLAYER1 wins) estimate: exactly 1 / 0 for a finished game; for a truncated one the value bgx_select_moves reports
 *              for the last ply played, or V(position, mover) as bgx_evaluate gives it when that ply had no sequence (or only the
 *              empty sequence of a blocked double);
 *   outcome    class of a finished trial from its final board: 1 / 2 / 3 PLAYER1 single / gammon (the loser bore nothing off) /
 *              backgammon (a gammon with a loser's checker on the bar or in the winner's home board), 4 / 5 / 6 the same for
 *              PLAYER2, 0 truncated.  Reported only: outcomes never change play or the mean.
 * Outputs, any may be NULL: mean[n] = sum x_t / trials, std_err[n] = sqrt(sum (x_t - mean)^2 / (trials (trials - 1))) (NaN for
 * one trial; with stratification this plain formula overestimates the error), both float64 and summed sequentially in trial
 * order; counts[n][8] = trials of outcome class 1..6, truncated trials, plies played in all trials.  The per-trial arrays
 * trial_value[n][trials], trial_outcome[n][trials], trial_plies[n][trials] are for analysis; without them the per-trial results
 * live in engine scratch.  A pure function of (position, mover, trials, max_plies, seed, flags, weights): batch composition,
 * order, chunking (bgx_set_option "rollout_chunk": trials per launch, rounded down to whole positions, 0 = 2^24) and warps per
 * CTA ("rollout_warps") change nothing.  BGX_E_INVALID for trials < 1, max_plies outside [0, BGX_ROLLOUT_MAX_PLIES], unknown
 * flags or a stratified rollout whose trials are not a multiple of 36.  The device form queues its work on the engine's stream;
 * the host form copies in, runs and copies out with one synchronisation. */
#define BGX_ROLLOUT_STRATIFY 1
#define BGX_ROLLOUT_MAX_PLIES 4096
int bgx_rollout(bgx_engine *e, const int8_t *positions, int64_t n, int32_t trials, int32_t max_plies, uint64_t seed, int flags,
                double *mean, double *std_err, int64_t *counts,
                float *trial_value, int8_t *trial_outcome, int32_t *trial_plies);
int bgx_rollout_host(bgx_engine *e, const int8_t *positions, int64_t n, int32_t trials, int32_t max_plies, uint64_t seed, int flags,
                     double *mean, double *std_err, int64_t *counts,
                     float *trial_value, int8_t *trial_outcome, int32_t *trial_plies);

/* The same call, asynchronous: copies and kernel are queued on lane `lane`'s own stream
 * (0 <= lane < BGX_ASYNC_LANES) and the call returns at once; bgx_lane_wait(lane) blocks until
 * that lane's outputs are in the host buffers.  Host buffers should be page-locked and must
 * stay untouched until the wait.  A lane holds one batch at a time (BGX_E_STATE otherwise).
 * With two or three lanes a host loop (model.py make_move callers: train.py:107, benchmark.py:86)
 * advances one part of its games while the GPU plays the others.  A lane's launch occupies half
 * the SMs, so the batches of two lanes are resident at once (a one-ply batch cannot be shorter
 * than its biggest turn tree; bgx_set_option "select_lane_grid" overrides the CTA count, 0 = every SM).
 * Batches of up to 2^21 queries ("select_order_max") are walked heaviest first: the order
 * never changes a result, only when it is computed. */
#define BGX_ASYNC_LANES 4
int bgx_select_moves_host_async(bgx_engine *e, int lane, const int8_t *queries, int64_t n, float epsilon, uint64_t seed,
                                int8_t *chosen, int8_t *moves, int8_t *moves_len, float *value,
                                int32_t *n_seq, int32_t *n_scored);
int bgx_lane_wait(bgx_engine *e, int lane);

/* One iteration of play_game's loop (train.py:103-121: make_move, is_game_over, setTurn, roll_dice) for n games,
 * host buffers in and out, asynchronous on `lane` like the call above.  records[i] = position, mover, the dice
 * already rolled.  next_records[i] = the chosen afterstate advanced exactly as bgx_advance_host does it: byte 31 =
 * 1 / 2 when the move ended the game, else 0 and the mover flipped; bytes 29,30 = the dice of ply next_ply[i] of game
 * game_id[i] (NULL: 0 / i) under dice_seed.  winner[i] = 0 / 1 / -1; winner, value, n_seq may be NULL.
 * Restarting finished games stays with the caller. */
int bgx_play_ply_host_async(bgx_engine *e, int lane, const int8_t *records, const int32_t *next_ply, const int64_t *game_id,
                            int64_t n, float epsilon, uint64_t explore_seed, uint64_t dice_seed,
                            int8_t *next_records, int8_t *winner, float *value, int32_t *n_seq);

/* The same loop iteration with the population's bookkeeping done on the device (train.py:199-220 / 527-547 run game after
 * game in every slot): ply[i] holds the ply number of records[i] and game_id[i] its game; on return they describe
 * next_records[i].  A game that ended is replaced IN PLACE by its slot's next game: id + id_stride, the opening position
 * (game.cpp:251), first mover by `first_mover` (BGX_FIRST_*), the dice of its ply 0; winner[i] still reports 0 / 1 for the
 * game that ended (-1 otherwise).  The caller's loop is submit / wait / swap buffers, nothing per game. */
int bgx_play_ply_restart_host_async(bgx_engine *e, int lane, const int8_t *records, int32_t *ply, int64_t *game_id, int64_t id_stride,
                                    int first_mover, int64_t n, float epsilon, uint64_t explore_seed, uint64_t dice_seed,
                                    int8_t *next_records, int8_t *winner, float *value, int32_t *n_seq);

/* The rest of a host-driven ply (train.py:113-121, benchmark.py:88-101) for n games at once, on
 * DEVICE buffers: next[i] = chosen[i] (an afterstate RECORD as bgx_select_moves writes it) with
 *   byte 31 = 1 / 2 when the move ended the game for PLAYER1 / PLAYER2 (game.cpp:388-407, PLAYER1
 *             is checked first), else 0 and the mover (byte 28) flipped,
 *   bytes 29,30 = the dice of ply `ply` of game game_id[i] (NULL: i) under the self-play dice rule
 *             (Philox key = seed, counter = (ply, id lo, id hi, 0)).
 * winner[i] (may be NULL) = 0 / 1 / -1.  next may alias chosen. */
int bgx_advance(bgx_engine *e, const int8_t *chosen, int8_t *next, int64_t n, uint64_t seed, int32_t ply,
                const int64_t *game_id, int8_t *winner);
/* The same on HOST buffers, for a host loop around bgx_select_moves_host[_async] whose games are not in
 * lockstep: ply[i] is the ply whose dice game i gets (the caller counts; NULL: 0), no engine needed. */
int bgx_advance_host(const int8_t *chosen, int8_t *next, int64_t n, uint64_t seed, const int32_t *ply,
                     const int64_t *game_id, int8_t *winner);
/* threads bgx_advance_host may use (0 = automatic: up to 4); several ranks sharing a box pass cores / ranks */
int bgx_set_host_threads(int n);

/* ------------------------------------------------------------------------------------
 * 4. Self-play population (replaces play_game, train.py:64-121, for many games at once)
 * ---------------------------------------------------------------------------------- */
typedef struct bgx_stats {
    int64_t plies;            /* plies played in this call (no-move plies included, train.py:103-121) */
    int64_t sequences;        /* legal turn sequences enumerated (reference-equivalent count) */
    int64_t scored;           /* afterstates scored by the MLP */
    int64_t games_finished;
    int64_t p1_wins;
    int64_t truncated;        /* games that hit traj_cap before ending */
    int64_t td_steps;         /* TD(lambda) steps replayed (bgx_td_replay) */
    double td_sq_error;       /* sum of td_error^2 over the non-terminal steps (train.py:162) */
    int64_t tree_edges;       /* moves applied while walking the turn trees (work actually done; <= what the reference walks) */
    int64_t td_live_rows;     /* TD replay: first-layer rows updated in the step passes (non-zero features of s_t, s_t+1, s_t+2), summed over the steps */
    int64_t td_lazy_row_steps;/* TD replay: (row, step) pairs replayed late, when a sleeping row re-entered the window or at the end of its game */
} bgx_stats;

/* first-mover rule */
#define BGX_FIRST_ROLLOFF 0   /* play_game's roll-off by dice sums, train.py:89-97 */
#define BGX_FIRST_PARITY 1    /* game id % 2, benchmark.py:74 / train.py:265 */

/* n_slots concurrent games.  Slot s plays global game ids first_id + s, then
 * + id_stride, + 2*id_stride ... (id_stride = global population, so sharding the slots
 * over ranks does not change any game).  Dice of ply p of game g are Philox4x32-10 with
 * key = seed and counter = (p, g_lo, g_hi, 0): d1 = 1 + ((x0*6)>>32), d2 likewise from x1
 * (replayable into the reference through Game.setDice, backgammon_bindings.cpp:86).
 * traj_cap > 0 records every pre-move RECORD (train.py:105-106) for bgx_td_replay. */
int bgx_selfplay_init(bgx_engine *e, int64_t n_slots, int64_t first_id, int64_t id_stride,
                      uint64_t seed, int first_mover, int32_t traj_cap);
/* also log the chosen afterstate of every ply (needed by bgx_export_trajectory's `chosen`;
 * off by default: it doubles the trajectory memory).  Call before bgx_selfplay_init. */
int bgx_selfplay_record_chosen(bgx_engine *e, int on);
/* every slot advances by n_plies plies; finished games restart in place with the next id */
int bgx_selfplay_step(bgx_engine *e, int32_t n_plies, float epsilon, bgx_stats *out);
/* every slot plays its current game to the end (or traj_cap), no restart: one "round" of
 * self-play from one weight snapshot (train.py:527-537) */
int bgx_selfplay_round(bgx_engine *e, float epsilon, bgx_stats *out);
/* start the next round: every slot gets its next game id and the opening position */
int bgx_selfplay_next_round(bgx_engine *e);

/* host copies of slot state: records[n_slots][32] (byte 28 = player to move, byte 31 =
 * 0 running / 1 PLAYER1 won / 2 PLAYER2 won), ply[n_slots], game_id[n_slots] */
int bgx_selfplay_read(bgx_engine *e, int8_t *records, int32_t *ply, int64_t *game_id);
/* trajectory of one slot's current game: pre[T][32] pre-move RECORDs with the dice rolled
 * (bytes 29,30), chosen[T][32] afterstates (byte 31 = sequence played flag); *T plies. */
int bgx_export_trajectory(bgx_engine *e, int64_t slot, int32_t cap, int8_t *pre, int8_t *chosen, int32_t *T);

/* records[n_slots * per_game][32]: `per_game` pre-move RECORDs (dice included) of every slot's current game, each taken at
 * a ply drawn uniformly from the plies recorded so far (Philox key = seed, counter = (j, slot lo, slot hi, 3)); all-zero
 * records for a slot with no recorded ply.  The "positions sampled from playouts at a uniform ply" of the enumeration
 * sweep (benchmark.py:64-96 plays such games with _random_move, benchmark.py:54-61).  Device / host buffer. */
int bgx_selfplay_sample(bgx_engine *e, int32_t per_game, uint64_t seed, int8_t *records);
int bgx_selfplay_sample_host(bgx_engine *e, int32_t per_game, uint64_t seed, int8_t *records);

/* ------------------------------------------------------------------------------------
 * 5. TD(lambda)  (replaces apply_td_updates, train.py:124-172)
 * ---------------------------------------------------------------------------------- */

/* Exact online TD(lambda) replay of every finished slot trajectory, each from the engine's
 * current weights (the round snapshot) with zeroed traces; the per-game weight changes are
 * SUMMED into delta[BGX_NPARAMS_PADDED] (device fp32, WEIGHTS order flattened: W1,b1,w2,b2;
 * overwritten, not accumulated).  Weights are not modified.  lr and lambda are doubles, as
 * model.learning_rate / model.lambda_decay are Python floats: lr * td_error is formed in
 * float64 and rounded to fp32 (train.py:147), lambda is rounded to fp32 when it meets the
 * trace tensor.  Trajectories of up to BGX_TD_MAX_STEPS recorded plies (traj_cap above that
 * is refused); out->truncated counts the slots skipped because their game hit traj_cap. */
#define BGX_TD_MAX_STEPS 2048
int bgx_td_replay(bgx_engine *e, double lr, double lambda, float *delta_dev, bgx_stats *out);
/* The same with the reference's PER-GAME schedule (train.py:538 calls update_learning_params(games_done + k + 1)
 * before replaying the k-th game of a round; model.py:69-73: lr = max(0.01, 0.1 * 0.96^(episode // 40000)),
 * lambda = max(0.7, 0.9 * 0.96^(episode // 30000))): the game in slot s of this engine is episode
 * games_done + first_id + s + 1, where first_id is the population's first global slot (bgx_selfplay_init) -
 * the k-th game of the round in global slot order. */
int bgx_td_replay_scheduled(bgx_engine *e, int64_t games_done, float *delta_dev, bgx_stats *out);
/* weights += scale * delta   (after the caller's allreduce over ranks) */
int bgx_apply_delta(bgx_engine *e, const float *delta_dev, float scale);
/* both in one call for a single-GPU caller: delta_host[BGX_NPARAMS] (may be NULL) receives the summed weight
 * change, then weights += scale * delta (scale 0: weights untouched).  One round of train.py:527-547. */
int bgx_td_round_host(bgx_engine *e, double lr, double lambda, float scale, float *delta_host, bgx_stats *out);
/* one external trajectory (host buffers): records[T][32] with byte 28 = the turn flag of each
 * pre-move state; new_* receive the weights after the replay; sq_errors[T-1] may be NULL */
int bgx_td_replay_host(bgx_engine *e, const int8_t *records, int32_t T, int player1_won,
                       double lr, double lambda,
                       float *new_W1, float *new_b1, float *new_w2, float *new_b2, double *sq_errors);

/* The cross-GPU exchange of a training round (replaces the pickling of trajectories back to the main process and its
 * sequential replay, train.py:330-348, 527-547): ONE all-reduce(sum) of the fp32[BGX_NPARAMS_PADDED] weight delta per round,
 * in place, on the engine's stream, through an NCCL communicator the caller owns (ncclComm_t; NCCL is bound with dlopen at
 * first use, libbgx does not link it).  Afterwards every rank calls bgx_apply_delta with the same buffer. */
int bgx_allreduce_delta(bgx_engine *e, void *nccl_comm, float *delta_dev);
/* For callers without an NCCL binding of their own: the three calls that make a communicator.  id128 is the 128-byte
 * ncclUniqueId that rank 0 creates and hands to the other ranks by any means (a file, MPI, torch.distributed, a socket).
 * bgx_nccl_load names the library explicitly (NULL / not called: "libnccl.so.2" by the loader's search path). */
int bgx_nccl_load(const char *libnccl_path);
int bgx_nccl_unique_id(void *id128);
int bgx_nccl_comm_init(bgx_engine *e, int n_ranks, int rank, const void *id128, void **nccl_comm);
int bgx_nccl_comm_destroy(void *nccl_comm);

/* ------------------------------------------------------------------------------------
 * 6. Introspection for benchmarks
 * ---------------------------------------------------------------------------------- */
/* kernels launched by this engine since creation (bench.py's gpu_launches) */
int bgx_launch_count(bgx_engine *e, int64_t *n);
/* CUDA-event duration (ms) of the last self-play / select / enumerate kernel launch */
int bgx_last_kernel_ms(bgx_engine *e, float *ms);
int bgx_device_props(bgx_engine *e, int *sm_count, int *clock_khz, int64_t *global_mem);
/* on != 0: later TD replays run the instrumented variant of k_td_replay.  cycles[8][16] (may be NULL) receives what the last
 * instrumented launch recorded on CTA 0, per warp (= row class): [0..7] SM cycles lane 0 spent in each phase of the step
 * (first-layer store, barrier, hidden layer, window bookkeeping + lazy replay, barrier, values + gradients, row pass, end of
 * game; a barrier's wait shows up in the phase that follows it), [15] the TD steps of that CTA. */
int bgx_td_profile(bgx_engine *e, int on, uint64_t *cycles);
/* Exhaustive device check of what the greedy ply's ranking relies on (bgx_ply.cuh PlyEvaluator::value_of; the reference ranks by
 * the value itself, model.py:205-213): ex2.approx.ftz is non-decreasing over every pair of neighbouring finite floats and
 * rcp.approx.ftz non-increasing over [1, FLT_MAX].  Both counts of violations must be 0 on the device in use. */
int bgx_sfu_monotone(bgx_engine *e, int64_t *ex2_violations, int64_t *rcp_violations);
/* warps per CTA of the fused ply kernels as configured */
int bgx_kernel_config(bgx_engine *e, int *selfplay_warps, int *select_warps);
/* tuning knobs of the fused ply kernels for benchmarks and probes; the defaults are the measured best.  Keys:
 * "selfplay_warps", "select_warps" (16, 20, 24, 32), "select_lane_grid", "select_order_max", "select_urgent_min",
 * "select_giant_min", "select_urgent_from_pct"; for bgx_select_moves_2ply "twoply_chunk" (replies per k_select launch, 0 = 2^21)
 * and "twoply_timing" (1: time its stages, synchronising between them).  The library reads no environment variables. */
int bgx_set_option(bgx_engine *e, const char *key, int64_t value);
/* stage times (ms) accumulated by two-ply calls under "twoply_timing" since the last read: [0] candidates (summary walk, scan,
 * candidate walk), [1] expansion filter and list, [2] replies (records + k_select), [3] expectation and pick; reset by the read */
int bgx_twoply_stage_ms(bgx_engine *e, double *ms);

#ifdef __cplusplus
}
#endif
#endif /* BGX_H */
