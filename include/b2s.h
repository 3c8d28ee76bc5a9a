/* b2s.h — C ABI of the B200-native batched game-simulation and search engine.
 *
 * This is the drop-in boundary for ONE hot path of google-deepmind/open_spiel: the per-game
 * State transition functions (ApplyAction / LegalActions / IsTerminal / Returns /
 * ObservationTensor) of tic_tac_toe, connect_four, breakthrough, hex, go, kuhn_poker and
 * leduc_poker, and the MCTSBot / CFRSolver loops that drive them.  Everything here runs as
 * hand-written sm_100a CUDA over struct-of-arrays batches of packed states resident in HBM.
 * There is no CPU fallback: every entry point fails (non-zero status) when no CUDA device exists.
 *
 * Shape follows the reference's own C-ABI precedent, open_spiel/go/go_open_spiel.h:21-70
 * (opaque handles, caller-allocated output buffers), extended with an error channel because a
 * batch call must not exit() the process the way SpielFatalError (spiel_utils.cc:119-135) does.
 *
 * Conventions
 *  - every function returns 0 on success, non-zero on failure; b2s_last_error() gives the message
 *    (thread-local).  Nothing throws, nothing calls exit().
 *  - "_d" pointers are DEVICE pointers on the batch's device, "_h" pointers are HOST pointers.
 *  - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream); calls with
 *    device pointers only enqueue work.  The *_host entry points copy, run and synchronise.
 *  - a batch is not thread-safe; distinct batches are independent.
 *  - actions are int32 (the reference's Action is int64, spiel_utils.h:134; all seven games have
 *    fewer than 2^15 distinct actions).  Action -1 (kInvalidAction, spiel_globals.h:82) means
 *    "leave this lane untouched" in batched calls — the reference has no batched call, so this is
 *    an extension; its own ApplyAction CHECKs action != -1 (spiel.cc:441-451).
 *  - an illegal action, or any action on a terminal state, leaves the lane unchanged and is counted;
 *    b2s_error_count() reports how many lanes were rejected since the last reset (the reference
 *    would have SPIEL_CHECK-aborted inside DoApplyAction, e.g. connect_four.cc:131-133).
 *  - returns are float32 on the device: every value the seven games can return (+-1, 0, -0, and
 *    Leduc's half-integers, Kuhn's small integers) is exactly representable, so widening to the
 *    reference's double (spiel.h:470) is bit-exact, sign of zero included.
 */
#ifndef B2S_H_
#define B2S_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- games ------------------------------------------------------------------------------- */

/* Replaces GameRegisterer::CreateByName lookup, open_spiel/spiel.cc:150-170.
 * Returns a small non-negative id for a supported short_name, -1 otherwise. */
int b2s_game_id(const char* short_name);
enum {
  B2S_TIC_TAC_TOE = 0, B2S_CONNECT_FOUR = 1, B2S_BREAKTHROUGH = 2, B2S_HEX = 3, B2S_GO = 4,
  B2S_KUHN_POKER = 5, B2S_LEDUC_POKER = 6, B2S_MNK = 7, B2S_OTHELLO = 8, B2S_Y = 9, B2S_HAVANNAH = 10, B2S_NUM_GAMES = 11
};

/* Game parameters (replaces GameParameters, open_spiel/game_parameters.h:31-120, for the seven
 * games).  Unset fields (< 0 / NaN) take the reference defaults. Names match the reference's
 * parameter_specification (e.g. connect_four.cc:50-54, go.cc:55-63, hex.cc:48-55). */
typedef struct b2s_params {
  int32_t rows;            /* connect_four, breakthrough; hex num_rows; mnk n */
  int32_t columns;         /* connect_four, breakthrough; hex num_cols; mnk m */
  int32_t x_in_row;        /* connect_four; mnk k */
  int32_t egocentric_obs_tensor; /* connect_four */
  int32_t board_size;      /* hex, go */
  int32_t swap;            /* hex */
  int32_t plain_obs_tensor;/* hex */
  int32_t handicap;        /* go */
  int32_t max_game_length; /* go */
  int32_t players;         /* kuhn_poker, leduc_poker (2 only on device) */
  int32_t starting_player; /* leduc_poker */
  int32_t reserved[5];
  double komi;             /* go */
  double reserved_d[3];
} b2s_params;
void b2s_params_default(b2s_params* p);   /* all fields "unset" */

/* What Game::{NumDistinctActions,NumPlayers,MaxGameLength,ObservationTensorSize,...} return
 * (open_spiel/spiel.h:927-1190), plus the batch layout facts a caller needs to size buffers. */
typedef struct b2s_game_info {
  int32_t game_id;
  int32_t num_players;
  int32_t num_distinct_actions;
  int32_t max_game_length;
  int32_t max_chance_outcomes;
  int32_t observation_tensor_size;
  int32_t information_state_tensor_size;   /* 0 when the game provides none */
  int32_t mask_words;                      /* ceil(max(num_distinct_actions, max_chance_outcomes)/32) */
  int32_t state_bytes;                     /* bytes of packed state per lane (excluding history) */
  int32_t history_bytes;                   /* extra per-lane bytes (go: superko hash history) */
  double min_utility, max_utility;
  int32_t obs_shape[4];                    /* ObservationTensorShape, zero padded */
  int32_t reserved[4];
} b2s_game_info;
int b2s_game_info_get(int game_id, const b2s_params* params, b2s_game_info* out);

/* ---- batches of states ------------------------------------------------------------------- */

/* A batch = `capacity` packed State objects (open_spiel/spiel.h:301-916) of one game, SoA in HBM. */
int  b2s_batch_create(int game_id, const b2s_params* params, int64_t capacity, int device, void** out_batch);
void b2s_batch_destroy(void* batch);
int  b2s_batch_info(void* batch, b2s_game_info* out);
int64_t b2s_batch_capacity(void* batch);

/* Game::NewInitialState (spiel.h:941) for lanes [0, n). Clears the error counter. */
int b2s_reset(void* batch, int64_t n, void* stream);

/* State::ApplyAction (spiel.cc:441-451) on lanes [0, n). */
int b2s_apply_actions(void* batch, const int32_t* actions_d, int64_t n, void* stream);

/* State::LegalActionsMask (spiel.cc:518-524) as bit masks: mask_words uint32 per lane, bit a of
 * word a/32 set iff action a is legal for the player to move (all zero at terminal states).  At a
 * chance node the mask holds the available chance outcomes. */
int b2s_legal_mask(void* batch, uint32_t* mask_words_d, int64_t n, void* stream);

/* State::LegalActions (spiel.h:388): ascending action ids, `stride` int16 slots per lane
 * (stride >= max legal count), counts_d[i] = number of legal actions of lane i. */
int b2s_legal_list(void* batch, int16_t* actions_d, int32_t* counts_d, int32_t stride, int64_t n, void* stream);

/* State::CurrentPlayer / IsTerminal / Returns (spiel.h:330,447,470).  Any output may be NULL.
 * current_player: >=0 player, -1 chance (kChancePlayerId), -4 terminal (kTerminalPlayerId).
 * returns_d is [n][num_players] float32; like every float output it needs 4-byte alignment only. */
int b2s_status(void* batch, int8_t* current_player_d, uint8_t* terminal_d, float* returns_d, int64_t n, void* stream);

/* State::ObservationTensor(player) (spiel.cc:908-925): [n][observation_tensor_size] float32,
 * CHW row-major as utils/tensor_view.h:32-54.  player = -1 observes as the player to move
 * (player 0 at terminal / chance nodes). */
int b2s_observation(void* batch, int player, float* obs_d, int64_t n, void* stream);
/* State::InformationStateTensor(player) (kuhn_poker, leduc_poker). */
int b2s_information_state(void* batch, int player, float* out_d, int64_t n, void* stream);

/* Fused env step: ApplyAction, then IsTerminal, Returns and the next LegalActionsMask in one pass
 * over the state.  Outputs may be NULL. */
int b2s_step_fused(void* batch, const int32_t* actions_d, uint32_t* mask_words_d, uint8_t* terminal_d,
                   float* returns_d, int64_t n, void* stream);
/* Same call with HOST buffers (pinned or pageable): copies actions in, runs, copies results out,
 * synchronises.  This is the end-to-end entry a CPU-side caller (the State adapter, an RL env
 * loop such as python/rl_environment.py:337-431) uses. */
int b2s_step_fused_host(void* batch, const int32_t* actions_h, uint32_t* mask_words_h, uint8_t* terminal_h,
                        float* returns_h, int64_t n);
/* The same env step with byte-wide I/O, for host-driven loops where PCIe bytes per lane are the cost (win / loss / draw
 * games: tic_tac_toe, connect_four, breakthrough, hex, go).  actions_h: action_bytes = 1 -> uint8 per lane, 0xFF = leave
 * the lane untouched; action_bytes = 4 -> int32, -1 = untouched.  status_h: one byte per lane,
 *   bit 7      IsTerminal (spiel.h:447)
 *   terminal:  bits 0-1 = outcome: 0 draw (Returns {0,0}), 1 player 0 won ({+1,-1}), 2 player 1 won ({-1,+1})
 *   otherwise: bits 0-6 = the next LegalActionsMask when num_distinct_actions <= 7 (connect_four up to 7 columns), else 0
 * mask_words_h (nullable): the full mask words as b2s_step_fused_host writes them, for games with more actions.
 * Same information as b2s_step_fused_host (the sign of a zero return is not carried), 2 B instead of 17 B per
 * connect_four lane.  Ordering of both *_host entry points: they run on library-owned BLOCKING streams, i.e. after work
 * already enqueued on the legacy default stream (stream = NULL) for this device and before later NULL-stream work; work the
 * caller has in flight on other streams must be synchronised by the caller first.  Both return after the results are in
 * the host buffers.
 * With PINNED host buffers and n >= 65536 the upload -> kernel -> download pipeline is captured once per (batch, buffers, n)
 * into a CUDA graph and replayed with one launch per call instead of five driver calls per chunk; up to 4 graphs are kept
 * per batch, least recently used evicted.  A buffer must
 * stay pinned for as long as it is used with the batch.  B2S_HOST_GRAPH=0 keeps the plain stream path, which pageable
 * buffers and small batches always take.  b2s_host_graph_launches() counts the graph replays of this process.
 * Byte-wide entry without mask words, pinned + device-mapped buffers (cudaHostAlloc / cudaHostRegister under unified
 * addressing — what torch's pin_memory() gives), both 16-byte aligned: no copy at all — the step kernel reads the action
 * bytes from host memory and writes the status bytes back itself (B2S_HOST_ZEROCOPY=0 disables; b2s_host_zero_copy_steps()
 * counts). */
int b2s_step_fused_host_compact(void* batch, const void* actions_h, int action_bytes, uint8_t* status_h,
                                uint32_t* mask_words_h, int64_t n);

/* Number of lanes whose action was rejected since the last b2s_reset (synchronises the stream);
 * first_bad_lane (nullable) receives the lowest-numbered such lane seen first, or -1. */
int b2s_error_count(void* batch, int64_t* count, int64_t* first_bad_lane, void* stream);

/* Scalar bridge for a host-side State adapter: raw packed lane `idx` (state_bytes + history_bytes). */
int b2s_state_get(void* batch, int64_t idx, void* host_blob, size_t cap);
int b2s_state_set(void* batch, int64_t idx, const void* host_blob, size_t len);
/* Copies lane `src` of `src_batch` into lanes [dst_begin, dst_begin+count) of `dst_batch` (Clone). */
int b2s_broadcast_state(void* dst_batch, int64_t dst_begin, int64_t count, void* src_batch, int64_t src, void* stream);

/* Lane-range State::Clone (spiel.h:740): dst[dst_begin+i] = src[src_begin+i], i in [0,count). */
int b2s_copy_states(void* dst_batch, int64_t dst_begin, void* src_batch, int64_t src_begin, int64_t count, void* stream);

/* Gather-clone: dst[i] = src[src_lanes_d[i]], i in [0,count) (State::Child fan-out, spiel.h:740-744). */
int b2s_gather_states(void* dst_batch, void* src_batch, const int64_t* src_lanes_d, int64_t count, void* stream);

/* Random playouts to terminal from every lane's current state (the inner loop of
 * RandomRolloutEvaluator::Evaluate, algorithms/mcts.cc:43-72, and of examples/benchmark_game.cc:32-115):
 * uniform over legal actions (and over chance outcomes) from a Philox4x32-10 counter stream keyed
 * by (seed, lane + lane_offset, ply).  The batch states are advanced in place to their terminal
 * states.  returns_d [n][num_players] float32 and plies_d [n] int32 (plies played) may be NULL. */
int b2s_rollout(void* batch, uint64_t seed, int64_t lane_offset, int64_t n, float* returns_d, int32_t* plies_d, void* stream);

/* ---- self-play trajectories ----------------------------------------------------------------- */

/* Replaces algorithms::RecordBatchedTrajectory (open_spiel/algorithms/trajectories.h:34-100,
 * trajectories.cc:98-200) with uniform-random policies (GetUniformPolicy) for n episodes at once, started from
 * every lane's current state and played to the end (the batch is left at the terminal states).  Only decision
 * nodes are recorded; chance nodes are sampled and applied in between (trajectories.cc:152-157).  The fields are
 * the BatchedTrajectory fields, TIME-MAJOR: row t of every array is step t of all n episodes (the reference's
 * [B][T] layout is the transposed view), padded like BatchedTrajectory::ResizeFields (trajectories.cc:62-96):
 * legal mask all ones, everything else 0.  Device pointers; any may be NULL.
 *   observations      [T][n][F] float32  State::InformationStateTensor() of the acting player when the game has one
 *                                        (the reference's include_full_observations), else ObservationTensor()
 *   legal_mask        [T][n][mask_words] uint32  State::LegalActionsMask as bits (bit a of word a/32)
 *   actions           [T][n] int32,  player_ids [T][n] int8,  valid [T][n] uint8,  next_is_terminal [T][n] uint8
 *   rewards           [n][num_players] float32  terminal Returns()
 *   lengths           [n] int32  recorded steps per episode
 * player_policies is not materialised: it is 1/popcount(legal_mask) on the legal actions (padding: 1).
 * T = max_unroll_length must cover the longest episode (0: game max_game_length); an episode still running after
 * T decisions is counted by b2s_error_count (the reference CHECK-fails, trajectories.cc:64-68).  Random stream:
 * Philox4x32-10 keyed by (seed, lane + lane_offset, step), see csrc/batch_kernels.cuh. */
typedef struct b2s_trajectory_out {
  float*    observations;
  uint32_t* legal_mask;
  int32_t*  actions;
  int8_t*   player_ids;
  uint8_t*  valid;
  uint8_t*  next_is_terminal;
  float*    rewards;
  int32_t*  lengths;
} b2s_trajectory_out;
int b2s_record_trajectories(void* batch, uint64_t seed, int64_t lane_offset, int64_t n, int32_t max_unroll_length,
                            const b2s_trajectory_out* out, void* stream);

/* ---- MCTS ---------------------------------------------------------------------------------- */

/* Replaces algorithms::MCTSBot (open_spiel/algorithms/mcts.h:149-230) with a RandomRolloutEvaluator
 * (mcts.h:97-111) for n independent search roots at once: one tree per root, UCT or PUCT selection, optional
 * MCTS-Solver, run entirely on the device.  Field meaning = the MCTSBot constructor arguments
 * (mcts.h:161-169): uct_c, max_simulations, solve, seed; n_rollouts = RandomRolloutEvaluator's.
 * Deterministic perfect-information games only (tic_tac_toe, connect_four, breakthrough, hex, go).
 * Every tree owns an arena of 16-byte nodes (24 bytes when n_rollouts is not a power of two); max_nodes_per_tree is the
 * reference's node budget with its garbage collection, max_nodes_total the physical arena size (0 = derived).  A tree
 * that cannot allocate stops and is counted by b2s_error_count.  Chance nodes in the tree, Dirichlet noise and custom
 * evaluators are not device features (the host adapters route such bots to the stock MCTSBot). */
enum { B2S_MCTS_UCT = 0, B2S_MCTS_PUCT = 1 };   /* UCTValue mcts.cc:90-101 / PUCTValue :103-112 (uniform prior, :74-87) */
typedef struct b2s_mcts_config {
  int32_t max_simulations;
  int32_t n_rollouts;
  int32_t solve;
  int32_t child_selection_policy;   /* ChildSelectionPolicy (mcts.h:148): B2S_MCTS_UCT or B2S_MCTS_PUCT */
  double uct_c;
  uint64_t seed;
  int64_t tree_index_offset;   /* tree i uses random stream (seed, i + tree_index_offset): shard roots across GPUs */
  int64_t max_nodes_total;     /* physical arena nodes over all trees (0 = size from max_nodes_per_tree / free memory) */
  int64_t max_nodes_per_tree;  /* MCTSBot::max_nodes_ = (max_memory_mb << 20) / sizeof(SearchNode) + 1 (mcts.cc:214; 80-byte
                                  SearchNode): when a tree's node count reaches it the tree is garbage-collected exactly as
                                  MCTSBot::GarbageCollect does (mcts.cc:441-482).  0 / 1 = never (max_memory_mb = 0) */
  double  max_wall_clock_time; /* seconds; > 0: a tree stops starting simulations once this much time has passed (mcts.cc:362-365) */
  int32_t* gc_runs_d;          /* nullable device output [n_trees]: collections performed per tree */
} b2s_mcts_config;
/* MCTSBot::MCTSearch (mcts.cc:353-467) from lanes [0, n_trees) of roots_batch.  Outputs (device):
 * visit_counts_d [n][A] int32 and total_reward_d [n][A] double = explore_count / total_reward of the root's
 * children by action id (0 for illegal actions); outcome_p0_d [n][A] float = proven outcome for player 0 or
 * NaN (nullable); best_action_d [n] = SearchNode::BestChild (mcts.cc:127-143), -1 for terminal roots;
 * sims_run_d [n] = simulations actually run (the search stops early when the root is proven) (nullable).
 * Synchronises `stream` before returning. */
int b2s_mcts_search(void* roots_batch, int64_t n_trees, const b2s_mcts_config* cfg, int32_t* visit_counts_d,
                    double* total_reward_d, float* outcome_p0_d, int32_t* best_action_d, int32_t* sims_run_d,
                    void* stream);
/* Arena nodes consumed by the last b2s_mcts_search on this batch (sum over trees of the arena high-water marks). */
int b2s_mcts_nodes_used(void* roots_batch, int64_t* nodes);

/* ---- CFR ----------------------------------------------------------------------------------- */

/* Replaces algorithms::CFRSolver / CFRPlusSolver (open_spiel/algorithms/cfr.h:312-357) for two-player
 * games with an information-state tensor (kuhn_poker, leduc_poker): the game tree is expanded once with
 * the batched kernels, regret / average-policy tables live on the device, and every
 * EvaluateAndUpdatePolicy (cfr.cc:263-282) runs inside one persistent kernel.  FP64, reference operation
 * order: tables match the reference bit for bit. */
enum { B2S_CFR_LINEAR_AVERAGING = 1, B2S_CFR_REGRET_MATCHING_PLUS = 2,   /* both = CFRPlusSolver */
       B2S_CFR_MCCFR_TABLES = 4 };   /* tables start at kInitialTableValues = 1e-6 (external_sampling_mccfr.h:59) */
typedef struct b2s_cfr_info {
  int32_t num_nodes, num_levels, num_infosets, num_entries;   /* entries = sum of legal actions over infosets */
  int32_t key_floats;                                         /* information-state tensor size */
  int32_t iteration;
  int32_t chance_nodes, decision_nodes, terminal_nodes;       /* cf. integration_tests/api_test.py:77-88 */
  int32_t reserved[3];
} b2s_cfr_info;
int  b2s_cfr_create(int game_id, const b2s_params* params, int flags, int device, void** out_solver);
void b2s_cfr_destroy(void* solver);
/* `iters` x CFRSolverBase::EvaluateAndUpdatePolicy, enqueued on `stream`. */
int  b2s_cfr_iterate(void* solver, int iters, void* stream);
int  b2s_cfr_info_get(void* solver, b2s_cfr_info* out);
/* The CFRInfoStateValuesTable (cfr.h:42-104) as flat host arrays: per-entry cumulative_regrets /
 * cumulative_policy / current_policy [num_entries], offsets [num_infosets+1], legal actions [num_entries],
 * acting player [num_infosets], and the information-state tensor of every infoset
 * [num_infosets][key_floats] as its key (the reference keys by InformationStateString; both identify the
 * same perfect-recall information state).  Any pointer may be NULL. */
int  b2s_cfr_export(void* solver, double* regrets_h, double* cum_policy_h, double* cur_policy_h, int32_t* offsets_h,
                    int32_t* legal_actions_h, int32_t* players_h, float* keys_h, void* stream);
/* Restore tables (checkpoint / resume; cfr.cc:699-781 DeserializeCFRSolver).  iteration < 0 keeps the counter. */
int  b2s_cfr_import(void* solver, const double* regrets_h, const double* cum_policy_h, const double* cur_policy_h,
                    int iteration, void* stream);
/* NashConv of the average policy (use_average != 0; CFRAveragePolicy, cfr.cc:104-125) or of the current policy,
 * computed on the device over the same flattened tree — replaces algorithms::NashConv / Exploitability
 * (tabular_exploitability.cc) for the CFR loop of examples/cfr_example.cc:37-46; exploitability = nash_conv / 2.
 * values_out (nullable): {best-response value p0, p1, on-policy value p0, p1}.  Synchronises `stream`. */
int  b2s_cfr_nash_conv(void* solver, int use_average, double* nash_conv_out, double* values_out, void* stream);
/* The pure best responses behind those values (TabularBestResponse::GetBestResponseActions, best_response.cc:194-228):
 * best_action_index_h[I] = the best responder's choice at information state I (I in b2s_cfr_export order; the responder is
 * the state's own player, responding to the other player's average / current policy) as an index into that state's
 * legal actions — first maximum of the counterfactual-reach-weighted child values.  values_out as above (nullable). */
int  b2s_cfr_best_response(void* solver, int use_average, int32_t* best_action_index_h, double* values_out, void* stream);
/* Device pointers of the three per-entry tables. */
int  b2s_cfr_tables(void* solver, double** regrets_d, double** cum_policy_d, double** cur_policy_d);
/* Multi-GPU CFR (the path's one real exchange step; SURVEY §8e).  One player-traversal of iteration `iteration`
 * (1-based, CFRSolverBase::iteration_) is split in two launches around an all-reduce:
 *   traverse_shard(player, iteration, rank, world) -> all-reduce(contribution buffer, sum) -> apply_deltas
 * Every rank evaluates reach/value for the whole tree; the regret / average-policy contribution of history slot k (one
 * value per action) is written by rank k mod world and as 0.0 by the others, so the all-reduce — x + 0 + ... + 0, exact in
 * any order — hands every rank every contribution, and apply_deltas adds them in the reference's DFS order
 * (cfr.cc:387-401): the tables are BIT-IDENTICAL to the single-GPU solver and to the reference for any world size.
 * Either the caller performs the all-reduce (the three calls below, buffer = b2s_cfr_delta_buffer, length =
 * b2s_cfr_delta_count doubles) or the library does (b2s_cfr_iterate_sharded). */
int  b2s_cfr_traverse_shard(void* solver, int player, int iteration, int shard, int num_shards, void* stream);
int  b2s_cfr_apply_deltas(void* solver, void* stream);
int  b2s_cfr_delta_buffer(void* solver, double** delta_d);
int  b2s_cfr_delta_count(void* solver, int64_t* count);
/* In-library exchange (NCCL over NVLink; NCCL is resolved with dlopen, the copy already loaded in the process wins).
 * b2s_nccl_unique_id: 128-byte ncclUniqueId created on one rank, to be handed to all ranks by the caller's own means.
 * b2s_cfr_comm_init creates a communicator owned by the solver; b2s_cfr_comm_adopt uses the caller's ncclComm_t.
 * b2s_cfr_iterate_sharded: `iters` x CFRSolverBase::EvaluateAndUpdatePolicy (cfr.cc:263-282) with traverse -> ncclAllReduce
 * -> apply enqueued back to back on a solver-owned stream (ordered after / before `stream`), 16 iterations per CUDA graph
 * launch — no host code between the steps.  Collective: every rank must make the same call.
 * b2s_cfr_allreduce_probe: device seconds of `count` back-to-back all-reduces of the buffer alone (the latency floor). */
int  b2s_nccl_unique_id(void* id128);
int  b2s_cfr_comm_init(void* solver, const void* id128, int rank, int world);
int  b2s_cfr_comm_adopt(void* solver, void* nccl_comm, int rank, int world);
int  b2s_cfr_iterate_sharded(void* solver, int iters, void* stream);
int  b2s_cfr_allreduce_probe(void* solver, int count, double* seconds);
int  b2s_cfr_set_iteration(void* solver, int iteration);

/* Replaces algorithms::ExternalSamplingMCCFRSolver (open_spiel/algorithms/external_sampling_mccfr.h:55-110,
 * AverageType::kSimple) on a solver created with B2S_CFR_MCCFR_TABLES: `iters` x RunIteration
 * (external_sampling_mccfr.cc:71-80).  Every (iteration, traverser) phase runs `traversals_per_update` independent
 * UpdateRegrets traversals (:124-186) in parallel, one thread each, all reading the tables as they stand at the start
 * of the phase; their regret / average-policy deltas are then added in a fixed, documented order (deterministic, FP64).  With
 * traversals_per_update = 1 this is exactly the reference's algorithm.  The uniform variates come from a
 * position-keyed Philox stream (seed, path hash, phase, traversal) instead of the reference's sequential
 * std::mt19937; oracle/algorithms/mccfr.cc implements both streams and ties the two together.
 * Synchronises `stream`; fails if a sampling step found sum(probabilities) <= z (the reference's
 * SpielFatalError in SampleActionIndex, cfr.cc:617-628). */
int  b2s_mccfr_external_iterate(void* solver, int iters, int traversals_per_update, uint64_t seed, void* stream);
/* ... with options.  B2S_MCCFR_FULL_AVERAGE = AverageType::kFull (external_sampling_mccfr.h:53-54): no averaging inside the
 * traversals; after the two traversal phases of every iteration one pass over the whole tree adds
 * reach[player](h) * regret-matching policy at every decision node (FullUpdateAverage, external_sampling_mccfr.cc:188-230). */
enum { B2S_MCCFR_FULL_AVERAGE = 1 };
int  b2s_mccfr_external_iterate_ex(void* solver, int iters, int traversals_per_update, uint64_t seed, int flags, void* stream);
/* Replaces algorithms::OutcomeSamplingMCCFRSolver (open_spiel/algorithms/outcome_sampling_mccfr.h:40-66; default uniform
 * policy, no baseline) on a solver created with B2S_CFR_MCCFR_TABLES: `iters` x RunIteration (outcome_sampling_mccfr.cc:
 * 60-67).  Every (iteration, player) phase runs `trajectories_per_update` independent SampleEpisode trajectories (:150-247) in
 * parallel against the tables as they stand at the start of the phase; their regret / average-policy deltas are added in the
 * same fixed order as the external-sampling solver's.  trajectories_per_update = 1 is exactly the reference's algorithm; the
 * uniform variates come from the position-keyed Philox stream oracle/algorithms/os_mccfr.cc restates.  Synchronises. */
int  b2s_mccfr_outcome_iterate(void* solver, int iters, int trajectories_per_update, uint64_t seed, double epsilon, void* stream);
/* The same phase split over GPUs, bit-identical to the single-GPU call: the 64 lanes of the fixed-order reduction are
 * the unit of sharding.  Every rank runs the traversals k with k mod 64 in [lane_begin, lane_end) of phase
 * (current iteration, player) and writes those lanes of partials_d [64][num_entries]; after the lanes of all ranks have
 * been gathered (NCCL all-gather) every rank calls b2s_mccfr_apply_partials, which runs the reduction tree, updates the
 * (replicated) tables and, after player 1, advances the iteration counter. */
int  b2s_mccfr_traverse_lanes(void* solver, int player, int traversals_per_update, uint64_t seed, int lane_begin, int lane_end,
                              double* partials_d, void* stream);
int  b2s_mccfr_apply_partials(void* solver, int player, const double* partials_d, void* stream);

/* ---- pinned host memory helpers (for the *_host entry points) ----------------------------- */
int  b2s_host_alloc(void** out, size_t bytes);
void b2s_host_free(void* p);
int  b2s_device_alloc(int device, void** out, size_t bytes);
void b2s_device_free(int device, void* p);
int  b2s_memcpy_h2d(int device, void* dst_d, const void* src_h, size_t bytes, void* stream);
int  b2s_memcpy_d2h(int device, void* dst_h, const void* src_d, size_t bytes, void* stream);
int  b2s_stream_synchronize(int device, void* stream);
int  b2s_device_count(void);
/* Pins the calling thread to the CPUs local to `device` (sysfs local_cpulist of its PCI function), so that pinned
 * buffers it allocates afterwards (b2s_host_alloc, first touch) and its copy submissions stay on the GPU's NUMA node.
 * n_cpus (nullable) receives the size of that CPU set. */
int  b2s_bind_host_to_device(int device, int* n_cpus);

/* Launch accounting: number of kernels this library has launched in this process. */
int64_t b2s_launch_count(void);
int64_t b2s_host_graph_launches(void);
int64_t b2s_host_zero_copy_steps(void);

const char* b2s_last_error(void);
const char* b2s_version(void);

#ifdef __cplusplus
}
#endif
#endif /* B2S_H_ */
