/* ngp.h -- C ABI of libngp.so: the B200-native population-evaluation hot path of
 * n00b001/neuro-genetic-pong-self-play.
 *
 * The reference has no FFI layer; its operator surface is the DEAP toolbox plus three
 * duck-typed objects (SURVEY.md section 8b).  Each entry point below names the reference
 * interface it replaces (file:line in the reference tree).
 *
 * Conventions: every function returns 0 on success or a negative ngp_status;
 * ngp_last_error() gives the message for the calling thread.  All pointers are caller
 * owned.  Pointers documented "device" are CUDA device pointers on the handle's GPU,
 * "host" are ordinary host pointers (the *_host entry points stage through pinned memory
 * and include the copies).  `stream` is a cudaStream_t passed as void* (NULL = default
 * stream).  One handle per GPU; a handle is not thread-safe; distinct handles are
 * independent.  No torch types appear here.
 */
#ifndef NGP_H
#define NGP_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NGP_MAX_LAYERS 8
#define NGP_FRAME_ROWS 210
#define NGP_FRAME_COLS 160
#define NGP_RAM_BYTES 128
#define NGP_GAMES_TO_PLAY 6          /* config.py:46 */

typedef enum {
    NGP_OK = 0,
    NGP_ERR_INVALID = -1,            /* bad argument */
    NGP_ERR_CUDA = -2,               /* CUDA runtime error (message has the detail) */
    NGP_ERR_UNSUPPORTED = -3,        /* e.g. network too wide for the fused rollout */
    NGP_ERR_EMULATOR = -4            /* an environment hit an illegal opcode / decimal mode */
} ngp_status;

/* actions as the reference's model.run() returns them: [0,0] [1,0] [0,1] */
enum { NGP_ACT_NONE = 0, NGP_ACT_UP = 1, NGP_ACT_DOWN = 2 };
/* retro save states used by the reference: default ('Start', 1 player vs the cartridge
 * robot, main.py:40) and 'Start.2P' (main.py:21,51) */
enum { NGP_STATE_START_1P = 0, NGP_STATE_START_2P = 1 };
/* 6507 core: the cartridge statically translated to CUDA (default, fastest) or the table-driven
 * interpreter (generic; also the verify-mode core of ngp_env_step) */
enum { NGP_CORE_TRANSLATED = 1, NGP_CORE_INTERPRETER = 0 };
/* opponent schedule of one evaluation */
enum {
    NGP_SCHEDULE_REFERENCE = 0,      /* main.py:33-58: bot, robot, score-bot, 3 x hall of fame */
    NGP_SCHEDULE_ROUND_ROBIN = 1     /* genome i (right) vs genome (i+k) mod N (left), k=1..games */
};

/* What one entry of the 16-entry gym-retro button vector (8 buttons per player: BUTTON, -, SELECT, RESET, UP, DOWN, LEFT,
 * RIGHT) does to the console.  Paddle p "up" lowers its resistance.  An environment made with players=1 (the cartridge
 * robot game, main.py:40) consumes only entries 0..7; FILTERED (main.py:23,55) cancels UP+DOWN / LEFT+RIGHT of one player.
 * Default map = the reference's own names (config.py:15-20, main.py:91-92): [0] RIGHT_PLAYER_START_BUTTON = fire of paddle 1
 * (the right player), [15] LEFT_PLAYER_START_BUTTON = fire of paddle 0, [4]/[5] = paddle 1 up/down, [6]/[7] = paddle 0
 * up/down, [2]/[10] = SELECT, [3]/[11] = RESET.  Which Stella event each retro button really raises is third-party
 * behaviour that cannot be checked without gym-retro (DESIGN.md "button map"); the map is data so it can be corrected. */
enum { NGP_BTN_NONE = 0, NGP_BTN_FIRE_P0 = 1 /* +p */, NGP_BTN_UP_P0 = 5 /* +2p = up, +2p+1 = down */, NGP_BTN_SELECT = 13,
       NGP_BTN_RESET = 14 };

/* Mirror of /root/reference/config.py (names kept) + network shape + schedule. */
typedef struct {
    int32_t n_layers;                        /* len(NETWORK_SHAPE), config.py:30-32 */
    int32_t nodes[NGP_MAX_LAYERS];           /* NETWORK_SHAPE */
    int32_t bias;                            /* BIAS, config.py:34 */
    int32_t games_to_play;                   /* GAMES_TO_PLAY, config.py:46 (<= 6 for the reference schedule) */
    int32_t win_score;                       /* WIN_SCORE, config.py:53 */
    int32_t timeout_thresh;                  /* TIMEOUT_THRESH, config.py:28 */
    int32_t schedule;                        /* NGP_SCHEDULE_* */
    int32_t max_frames;                      /* 0 = unlimited; hard stop per episode (tests) */
    float time_scaler;                       /* TIME_SCALER, config.py:54 */
    float scaled_paddle_height;              /* SCALED_PADDLE_HEIGHT, config.py:10 */
    uint8_t ball_colour[3];                  /* BALL_COLOUR, config.py:4 */
    uint8_t left_colour[3];                  /* LEFT_GUY_COLOUR, config.py:5 */
    uint8_t right_colour[3];                 /* RIGHT_GUY_COLOUR, config.py:6 */
    uint8_t pad_[3];
    /* GA rates, config.py:36-43, 49-50 */
    float cxpb, cx_alpha, mutpb, mut_mu, mut_sigma, mut_indpb;
    int32_t tournament_size;                 /* TOURNAMENT_SIZE = POPULATION_SIZE // 4 */
    int32_t core;                            /* 6507 core of the fused rollout: NGP_CORE_* */
    uint8_t button_map[16];                  /* NGP_BTN_* per gym-retro button (see above) */
} ngp_config;

typedef struct ngp_handle ngp_handle;

/* Fills cfg with config.py's defaults for a population of `population` genomes. */
void ngp_default_config(ngp_config *cfg, int32_t population);
/* sizeof(ngp_config) of the library: a binding asserts its own struct against it before calling ngp_create */
int32_t ngp_config_size(void);
const char *ngp_last_error(void);
const char *ngp_version(void);

/* rom: the 2048-byte cartridge image (host).  Builds the power-on -> 'Start'/'Start.2P'
 * snapshots on the device with the CUDA core itself. */
int ngp_create(const ngp_config *cfg, const uint8_t *rom, int32_t device, ngp_handle **out);
int ngp_destroy(ngp_handle *h);
int32_t ngp_gene_size(const ngp_handle *h);                 /* utils.calculate_gene_size, utils.py:128-136 */

/* ---- K1: batched Atari 2600 core, explicit-action stepping (verify / stepwise mode) ----
 * Replaces retro.make + env.reset (main.py:21,40,51,56) and env.step (main.py:77). */
int ngp_env_reset(ngp_handle *h, int32_t n_envs, int32_t state_id, void *stream);
/* actions: device u8[n_envs][16] in gym-retro button order (config.py:15-23).  Outputs
 * (device, any may be NULL): ram u8[n][128]; frames u8[n][210][160][3] RGB (obs.npy layout);
 * loc f32[n][3][2] + valid u8[n][3]: the fused find_stuff result for the same frame;
 * regs u8[n][8] = A X Y SP P PCL PCH err. */
int ngp_env_step(ngp_handle *h, const uint8_t *actions, uint8_t *ram, uint8_t *frames,
                 float *loc, uint8_t *valid, uint8_t *regs, void *stream);
/* same, choosing the 6507 core explicitly (parity tests run both) */
int ngp_env_step_core(ngp_handle *h, int32_t core, const uint8_t *actions, uint8_t *ram, uint8_t *frames,
                      float *loc, uint8_t *valid, uint8_t *regs, void *stream);
/* debug/parity: TIA digest u32[n][8] (collision latches, object positions, paddle charges) */
int ngp_env_digest(ngp_handle *h, uint32_t *digest, void *stream);

/* ---- K2: frame -> observation.  Replaces utils.find_stuff / get_rect_quickly
 * (utils.py:14-19, 60-68).  frames: device u8[n][210][160][3]; loc f32[n][3][2] (row, col in
 * cropped coordinates; ball, left, right); valid u8[n][3] (0 == the reference's None). */
int ngp_find_stuff(ngp_handle *h, const uint8_t *frames, int32_t n, float *loc, uint8_t *valid, void *stream);

/* ---- K3: per-genome grouped MLP forward.  Replaces NeuralNetwork.__init__/populate_weights/
 * run (numpy_nn.py:35-69, 120-137).  genomes f32[n_genomes][G] (reference gene order, bias
 * weight = last column), x f32[n_genomes][envs][n_in]; act u8[n_genomes][envs] (NGP_ACT_UP/DOWN),
 * out (may be NULL) f32[n_genomes][envs][n_out]. */
int ngp_mlp_forward(ngp_handle *h, const float *genomes, const float *x, int32_t n_genomes, int32_t envs,
                    uint8_t *act, float *out, void *stream);

/* Two-call form for a genome set that is used for many forward passes (the reference builds a NeuralNetwork once per
 * individual -- __init__/populate_weights, numpy_nn.py:35-69, main.py:29 -- and calls run() every frame):
 * ngp_mlp_prepare re-lays the wide hidden layers of `genomes` out once (handle-owned copy; a snapshot, like the reference's
 * populate_weights: later changes to `genomes` are not seen), ngp_mlp_forward_prepared then streams those weights from HBM
 * straight into tensor memory.  Same arguments and results as ngp_mlp_forward; genomes / n_genomes must be the prepared ones. */
int ngp_mlp_prepare(ngp_handle *h, const float *genomes, int32_t n_genomes, void *stream);
int ngp_mlp_forward_prepared(ngp_handle *h, const float *genomes, const float *x, int32_t n_genomes, int32_t envs,
                             uint8_t *act, float *out, void *stream);

/* ---- fused hot path: population genomes in -> fitness out.  Replaces
 * toolbox.map(toolbox.evaluate, population) (ga.py:83, main.py:28-66, main.py:69-154).
 * genomes: device f32[n][G].  hof_genomes f32[n_hof][G], hof_fitness f64[n_hof] (device; may be
 * NULL with n_hof = 0).  hof_pick: optional device i32[n][3] (injected hall-of-fame choices for
 * games 3..5; NULL = drawn from Philox(seed, generation)).  Outputs (device): fitness f64[n];
 * rewards f64[n][games] (may be NULL); frames i32[n][games] (may be NULL).  *frames_total (host,
 * may be NULL) receives the number of emulated frames after the stream is synchronised. */
int ngp_evaluate(ngp_handle *h, const float *genomes, int32_t n, const float *hof_genomes,
                 const double *hof_fitness, int32_t n_hof, const int32_t *hof_pick, uint64_t seed,
                 uint64_t generation, double *fitness, double *rewards, int32_t *frames,
                 uint64_t *frames_total, void *stream);
/* Same through HOST buffers: copies genomes (and HoF) in and fitness out, synchronises. */
int ngp_evaluate_host(ngp_handle *h, const float *genomes, int32_t n, const float *hof_genomes,
                      const double *hof_fitness, int32_t n_hof, uint64_t seed, uint64_t generation,
                      double *fitness, uint64_t *frames_total);

/* left-player codes of ngp_play_matches that are not genome rows */
enum { NGP_OPP_HARDCODED = -1,         /* dumb_ais.HardcodedAi: game 0 of main.evaluate */
       NGP_OPP_SCORE_HARDCODED = -2,   /* dumb_ais.ScoreHardcodedAi: game 2 */
       NGP_OPP_ROBOT = -3 };           /* the cartridge robot game: game 1 ('Start', players=1, HardcodedAi on action[6:8]) */

/* ---- an explicit match list in one fused launch.  Generalises main.evaluate's schedule (main.py:28-66): cross tables
 * between generations, every genome against the scripted opponents, custom tournaments.
 * genomes: device f32[n_genomes][G]; right, left: device i32[n_matches].  Match m is one perform_episode
 * (main.py:69-112): genome row right[m] plays on the right; left[m] is a genome row, which plays on the left with the
 * x-mirrored inputs as in self-play, or an NGP_OPP_* code.  mult: optional device f64[n_matches], the hall-of-fame
 * multiplier on the right player's score bonus (calculate_reward, utils.py:104-109); NULL = 1.0.
 * Outputs (device): rewards f64[n_matches], the right player's reward by ngp_evaluate's formula; frames i32[n_matches]
 * (env.step calls, may be NULL); scores i32[n_matches][2] = (score1, score2) as the cartridge keeps them (RAM $8D, $8E),
 * i.e. the left and the right player's points (may be NULL).  The fall-back random actions of get_actions are keyed by
 * Philox(seed, generation, m, frame, player): ngp_evaluate's key with environment index = match index.  win_score,
 * timeout_thresh, max_frames, time_scaler, paddle height, colours, button map and core come from the handle's config;
 * schedule, games_to_play and the hall of fame play no part.  *frames_total (host, may be NULL) and the emulator-error
 * report behave as in ngp_evaluate.
 * A right[m] outside [0, n_genomes), a left[m] that is neither a row nor an NGP_OPP_* code, or n_matches < 1 return
 * NGP_ERR_INVALID and nothing is played: the lists are checked on the device and the count of bad entries is read back,
 * so the call synchronises its stream once before the rollout is launched.  Networks wider than the fused rollout
 * takes (any layer > 32 units) return NGP_ERR_UNSUPPORTED; ngp_play_matches_stepwise plays them. */
int ngp_play_matches(ngp_handle *h, const float *genomes, int32_t n_genomes,
                     const int32_t *right, const int32_t *left, const double *mult, int32_t n_matches,
                     uint64_t seed, uint64_t generation,
                     double *rewards, int32_t *frames, int32_t *scores,
                     uint64_t *frames_total, void *stream);

/* One frame of a recorded match (ngp_record_matches): what perform_episode saw and decided on env.step t
 * (main.py:76-107).  Enough to re-render the game pixel for pixel through ngp_env_step, and the raw material of
 * behaviour statistics (paddle-ball distance, action mix, fall-back frames, rally lengths). */
typedef struct {
    float   loc[3][2];   /* find_stuff after env.step t: (row, col) of ball, left, right in cropped coordinates; 0 when not
                          * found.  The rollout's FP64 centroid rounded to float, exactly as ngp_env_step rounds its loc */
    uint8_t valid;       /* bit 0 ball, bit 1 left paddle, bit 2 right paddle found */
    uint8_t score[2];    /* RAM $8D, $8E after env.step t (score1 = left, score2 = right) */
    uint8_t act;         /* the decisions taken on frame t, after the bounds clamp: left | right << 2 (NGP_ACT_*); they
                          * drive env.step t+1 */
    int32_t timeout;     /* calculate_timeout_and_frames' counter after frame t (main.py:128-135) */
} ngp_frame_record;      /* 32 bytes */

/* ---- ngp_play_matches with a per-frame trace of every match, recorded inside the same fused launch.
 * Every argument of ngp_play_matches means what it means there, and with key == NULL rewards, frames, scores and
 * *frames_total are bit-identical to ngp_play_matches on the same arguments.
 * record: device ngp_frame_record[n_matches][max_record], 16-byte aligned.  For t < min(frames[m], max_record) entry
 * m * max_record + t describes env.step t of match m; entries past that are left untouched.  frames[m] always holds the
 * full length, so a truncated record can be recognised.
 * key: optional device i32[n_matches], the environment index of the fall-back key Philox(seed, generation, key[m], frame,
 * player); NULL = m.  With it one match reproduces one game of an ngp_evaluate call exactly: round-robin game k of genome
 * g has key g * games + k.
 * Refusals (NGP_ERR_INVALID, nothing written): those of ngp_play_matches, max_record < 1, a NULL or misaligned record, and
 * any key[m] < 0 (counted on the device with the list check, no further synchronisation).  Networks wider than 32 units
 * return NGP_ERR_UNSUPPORTED; ngp_play_matches_stepwise records them. */
int ngp_record_matches(ngp_handle *h, const float *genomes, int32_t n_genomes,
                       const int32_t *right, const int32_t *left, const double *mult, const int32_t *key, int32_t n_matches,
                       uint64_t seed, uint64_t generation, int32_t max_record, ngp_frame_record *record,
                       double *rewards, int32_t *frames, int32_t *scores, uint64_t *frames_total, void *stream);

/* ---- save states (ALE cloneState/restoreState, gym-retro env.em.get_state()/set_state()).
 * One game state: the console (TIA, RIOT, paddles, CPU registers, RAM) and, when it was captured inside a match, the
 * episode (perform_episode's locals, main.py:70-75: frame counter, timeout, total_frames, last scores, last ball and the
 * decisions that drive the next env.step).  The contents are documented (DESIGN.md section 4, "save states") but opaque to
 * callers: state arrays are device memory, 16-byte aligned, and the library only reads states that carry the magic and
 * version of this format, the hash of the handle's cartridge image, players 1 or 2 and a matching checksum. */
#define NGP_GAME_STATE_BYTES 512
typedef struct { uint8_t b[NGP_GAME_STATE_BYTES]; } ngp_game_state;

/* out: device ngp_game_state[n_envs] <- the stepwise environments as ngp_env_reset / ngp_env_step left them (no episode). */
int ngp_env_get_state(ngp_handle *h, ngp_game_state *out, void *stream);
/* The counterpart of ngp_env_reset: the n_envs stepwise environments become the consoles of `states` (device, any episode
 * part is ignored).  The states' players value (gym-retro `players`: 1 for the cartridge robot game) must be the same for all.
 * The states are validated on the device and the count of bad ones is read back (the call synchronises its stream once); on
 * any bad state the call returns NGP_ERR_INVALID and the environments are left as they were. */
int ngp_env_set_state(ngp_handle *h, const ngp_game_state *states, int32_t n_envs, void *stream);

/* ---- ngp_record_matches whose matches may start from saved states and capture their own.
 * genomes .. key, seed, generation and the outputs mean what they mean in ngp_record_matches.
 * start: optional device i32[n_matches]; match m starts from states[start[m]] (device ngp_game_state[n_states]); -1 or
 *   start == NULL = the built-in start state ngp_play_matches picks.  The plan (players, multiplier) comes from the lists.
 * A state with an episode and fresh == 0 resumes that episode: frame counter (so frames[m] is the whole episode's length and
 *   the fall-back draws, keyed by frame, continue), timeout, total_frames, last scores, last ball and the decisions taken on
 *   the captured frame, which drive the first resumed env.step.  Resuming a capture with the same genomes, key, seed and
 *   generation gives the uninterrupted game's reward, frames, scores and record entries.
 * fresh != 0, or a state without an episode: a new perform_episode from that console (frame 0, no last score or ball,
 *   BLANK_ACTION first), as retro.make(state=...) would; points already in RAM count.
 * capture_at: optional device i32[n_matches] with capture device ngp_game_state[n_matches]: after capture_at[m] env.steps
 *   counted from the episode's start (0 = before the first) the state of match m, console and episode, is written to
 *   capture[m] -- only while the episode is still running, otherwise capture[m] is left untouched (frames[m] <= capture_at[m]).
 * record: as in ngp_record_matches (entry t = env.step t from the episode's start, so a resumed match writes entries at or
 *   after its start frame only), or NULL for none.  *frames_total counts the env.steps emulated in this call.
 * Refusals (NGP_ERR_INVALID, nothing written, one synchronisation as in ngp_play_matches): those of ngp_record_matches (with
 * a non-NULL record), start[m] outside [-1, n_states), a state that fails validation, a state whose players value disagrees
 * with left[m] (players 1 with NGP_OPP_ROBOT only), capture_at[m] < 0, capture_at without capture, misaligned state arrays.
 * Networks wider than 32 units return NGP_ERR_UNSUPPORTED (ngp_play_matches_stepwise below plays them).  With start,
 * capture_at and record all NULL the results are ngp_play_matches' bits. */
int ngp_play_matches_states(ngp_handle *h, const float *genomes, int32_t n_genomes,
                            const int32_t *right, const int32_t *left, const double *mult, const int32_t *key, int32_t n_matches,
                            const ngp_game_state *states, int32_t n_states, const int32_t *start, int32_t fresh,
                            const int32_t *capture_at, ngp_game_state *capture,
                            int32_t max_record, ngp_frame_record *record,
                            uint64_t seed, uint64_t generation, double *rewards, int32_t *frames, int32_t *scores,
                            uint64_t *frames_total, void *stream);

/* ---- ngp_play_matches_states on the per-frame driver, for networks of any width.
 * Takes ngp_play_matches_states' arguments in the same order and has its contract: the same outputs, the same record and
 * capture semantics, the same refusals (NGP_ERR_INVALID, nothing written) with the same single read-back before anything is
 * played.  Every match is played by the per-frame driver of wide ngp_evaluate: one launch per frame emulates every running
 * match, the networks run between the frames, one more launch decides.
 * Wide networks (any layer > 32 units): 6 inputs and at most 8 outputs as in ngp_evaluate, otherwise NGP_ERR_INVALID.  Every
 *   MLP side of every match is one row per frame; the rows are grouped by genome into chunks of T rows (T = the smallest power
 *   of two in [16, 128] not below the mean rows per genome that plays), and the chunks run through ngp_evaluate's wide MLP
 *   kernels with each chunk's genome as the weight index.  The whole genome table is packed once per call as ngp_mlp_prepare
 *   packs it (about 1.05 MB per genome for [6,512,512,2]).
 * Networks the fused rollout takes: the decisions are its FP64 policies, so rewards, frames, scores, records, captures and
 *   *frames_total are the fused entry points' bits on the same arguments.
 * The call returns after every match has finished: like wide ngp_evaluate it synchronises its stream every 8 frames. */
int ngp_play_matches_stepwise(ngp_handle *h, const float *genomes, int32_t n_genomes,
                              const int32_t *right, const int32_t *left, const double *mult, const int32_t *key, int32_t n_matches,
                              const ngp_game_state *states, int32_t n_states, const int32_t *start, int32_t fresh,
                              const int32_t *capture_at, ngp_game_state *capture,
                              int32_t max_record, ngp_frame_record *record,
                              uint64_t seed, uint64_t generation, double *rewards, int32_t *frames, int32_t *scores,
                              uint64_t *frames_total, void *stream);

/* ---- match sessions: a match list that the caller advances one env.step at a time, with seats whose decisions the caller
 * supplies.  The reference's perform_episode (main.py:69-112) takes any object with .run(vec6) -> [up, down] as a player
 * (a NeuralNetwork, a dumb_ais bot, human_control.HumanInput: SURVEY.md section 8b); NGP_PLAYER_EXTERNAL is such a player
 * outside the library -- a policy of another framework, a person, any controller.
 *
 * NGP_PLAYER_EXTERNAL, as right[m] or left[m] of a session's list, is a model in perform_episode's sense: its decision is
 * consumed only on the frames on which get_actions calls the models (ball and both paddles found); on other frames the
 * fall-back random or none action is played with the usual Philox key; the bounds clamp applies to it; timeout, termination,
 * reward, scores, records and captures are what ngp_play_matches_stepwise computes.  An external right seat may face a genome
 * row, an NGP_OPP_* code or NGP_OPP_ROBOT; an external left seat a genome row or an external right seat.  Only the session
 * entry points accept the code: every other match-list entry point refuses it. */
enum { NGP_PLAYER_EXTERNAL = -4 };
/* bits of a session's per-match flags */
enum { NGP_SESSION_NEED = 1,            /* the next step consumes this match's external decisions */
       NGP_SESSION_DONE = 2,            /* the match has ended (for good: the bit stays set) */
       NGP_SESSION_EMULATOR_ERROR = 4 };/* it ended on an emulator error */

typedef struct ngp_session ngp_session;

/* Begins a session over a match list and plays its env.step 0.
 * genomes .. generation, rewards, frames and scores mean what they mean in ngp_play_matches_stepwise (networks of any width;
 * genomes may be NULL with n_genomes == 0 when no seat names a row).  The refusals are that call's (NGP_ERR_INVALID, nothing
 * written, no session created), with NGP_PLAYER_EXTERNAL allowed as above, after the same single read-back of the list check.
 * obs: device f32[n_matches][2][6] and flags: device u8[n_matches], written by begin and by every step:
 *   flags[m]: NGP_SESSION_* bits.  On a step that sets NEED, obs[m][0] (left seat) and obs[m][1] (right seat) of an external seat
 *   hold utils.inference's vector (utils.py:139-153) exactly as a genome in that seat would get it, the left seat's x-mirrored as
 *   in self-play; the rows of the other seats are unspecified.
 * scores (may be NULL) holds the (left, right) points of the last decided frame after every step, the final points at the end.
 * The session owns its per-match state, MLP rows and counters: other calls on the handle between two steps (ngp_evaluate,
 * ngp_play_matches*, another session) do not disturb it.  Wide networks share the handle's packed weight copy
 * (ngp_mlp_prepare): a step re-packs the session's genome table when another call replaced it.
 * Every device array passed to begin is read or written by later steps and must stay valid and unchanged (genomes, lists, mult,
 * key, states) until ngp_session_end.  *out receives the session. */
int ngp_session_begin(ngp_handle *h, const float *genomes, int32_t n_genomes,
                      const int32_t *right, const int32_t *left, const double *mult, const int32_t *key, int32_t n_matches,
                      const ngp_game_state *states, int32_t n_states, const int32_t *start, int32_t fresh,
                      int32_t max_record, ngp_frame_record *record, uint64_t seed, uint64_t generation,
                      double *rewards, int32_t *frames, int32_t *scores, float *obs, uint8_t *flags,
                      void *stream, ngp_session **out);
/* One env.step of every running match: (1) the decisions of the frame just observed, the external seats' from actions (device
 * u8[n_matches][2], (left, right) NGP_ACT_*; entries of other seats are ignored, a consumed value outside 0..2 is played as
 * NGP_ACT_NONE and counted), (2) the record entry, the scores and, for a match that ends, its reward and frame count,
 * (3) with capture (device ngp_game_state[n_matches], 16-byte aligned, or NULL) the state of every match still running --
 * the state ngp_play_matches_states writes with capture_at[m] = its frame count at that point, (4) the env.step, (5) the wide
 * MLP rows of the next decisions.  Neither synchronises, allocates nor reads back (a wide step after another call replaced the
 * packed weights re-packs them first), so the caller's policy can run on the same stream between steps, and steps can be
 * captured into a CUDA graph.  A step after every match has ended changes no output. */
int ngp_session_step(ngp_session *s, const uint8_t *actions, float *obs, uint8_t *flags, ngp_game_state *capture, void *stream);
/* Synchronises the stream.  *running (may be NULL) = the matches still running, *frames_total (may be NULL) = the env.steps
 * emulated so far (ngp_play_matches_stepwise's *frames_total once every match has ended).  Returns NGP_ERR_EMULATOR if a
 * match stopped on an emulator error, NGP_ERR_INVALID if out-of-range actions were consumed (the message has the count). */
int ngp_session_status(ngp_session *s, int32_t *running, uint64_t *frames_total, void *stream);
/* Frees the session (waits for its work first).  ngp_destroy ends every session still open on the handle. */
int ngp_session_end(ngp_session *s);

/* ---- K4: GA step.  Replaces toolbox.select / varAnd(mate, mutate) inside eaSimple
 * (ga.py:89-94, main.py:165-170; DEAP selTournament, cxBlend, mutGaussian).
 * Injected noise (all device, all optional = NULL -> Philox(seed, generation)). */
typedef struct {
    const int32_t *sel_draws;     /* [n][tournament_size] aspirant indices */
    const uint8_t *cx_do;         /* [n/2] */
    const float *cx_u;            /* [n/2][G] uniforms in [0,1) */
    const uint8_t *mut_do;        /* [n] */
    const float *mut_u;           /* [n][G] uniforms */
    const float *mut_z;           /* [n][G] standard normals */
} ngp_noise;
/* genomes f32[n][G], fitness f64[n] -> next f32[n][G], parent_idx i32[n] (selection winners),
 * invalid u8[n] (1 = needs re-evaluation), stats f64[4] = avg std min max of fitness (main.py:158-162). */
int ngp_ga_step(ngp_handle *h, const float *genomes, const double *fitness, int32_t n, uint64_t seed,
                uint64_t generation, const ngp_noise *noise, float *next, int32_t *parent_idx,
                uint8_t *invalid, double *stats, void *stream);
/* population init: each gene uniform [0,1) (ga.py:85-87) from Philox(seed) */
int ngp_init_population(ngp_handle *h, float *genomes, int32_t n, uint64_t seed, void *stream);

/* toolbox.select / toolbox.mate / toolbox.mutate as separate callables (ga.py:89-94), the same arithmetic and the same
 * Philox streams as ngp_ga_step.
 * ngp_select: DEAP selTournament(individuals, k, tournsize = cfg.tournament_size): fitness f64[n] -> parent_idx i32[k];
 *   draws: optional device i32[k][tournsize] aspirant indices (NULL = Philox(seed, generation)).  Without injected draws
 *   and from 8192 aspirants per tournament upwards the winners are drawn from the tournament's order statistics on the
 *   fitness-sorted population (one uniform per slot, ties uniform inside the tie group): the same distribution as
 *   tournsize draws per slot, in O(N log^2 N) instead of O(N * tournsize).
 * ngp_mate: DEAP cxBlend(ind1, ind2, cfg.cx_alpha) in place on two device genomes f32[G]; u: optional device f32[G]
 *   uniforms (NULL = the Philox stream of pair `pair`).
 * ngp_mutate: DEAP mutGaussian(ind, mu, sigma, indpb) in place; u / z: optional device f32[G] uniforms / standard normals
 *   (NULL = the Philox streams of individual `slot`). */
int ngp_select(ngp_handle *h, const double *fitness, int32_t n, int32_t k, const int32_t *draws, uint64_t seed,
               uint64_t generation, int32_t *parent_idx, void *stream);
int ngp_mate(ngp_handle *h, float *ind1, float *ind2, const float *u, int32_t pair, uint64_t seed, uint64_t generation,
             void *stream);
int ngp_mutate(ngp_handle *h, float *ind, const float *u, const float *z, int32_t slot, uint64_t seed, uint64_t generation,
               void *stream);

/* ---- hall of fame.  Replaces DEAP tools.HallOfFame(maxsize).update(population) (ga.py:78, main.py:165-168;
 * consumed by utils.create_model_from_hall_of_fame, utils.py:90-101).  Device resident and caller owned:
 * hof_genomes f32[maxsize][G] and hof_fitness f64[maxsize] hold the members best first in their first *n_hof rows.
 * Individuals are visited in population order; one enters when the hall is not full or its fitness is strictly above the
 * current worst, unless its genes equal a member's (64-bit hash, full compare on a hash match); a full hall drops its worst
 * first; the newcomer goes BEFORE members of equal fitness (DEAP's bisect_right on the ascending key list).
 * n_hof (host, in/out): member count.  The call synchronises the stream. */
int ngp_hof_update(ngp_handle *h, float *hof_genomes, double *hof_fitness, int32_t *n_hof, int32_t maxsize,
                   const float *genomes, const double *fitness, int32_t n, void *stream);

/* ---- multi-GPU exchange, device side (the reference's toolbox.map = scoop.futures.map gathers every fitness on the
 * master and eaSimple updates one hall of fame, ga.py:83, main.py:165-170).  One fixed-size record per rank travels in
 * the per-generation all-gather:
 *   [ n_local i32 | k_local i32 | 8 B pad | fitness f64[n_max] | elite_fitness f64[k_max] | elite_genomes f32[k_max][G] ]
 * (ngp_exchange_bytes, a multiple of 16; shards may differ in size when the population does not divide by the world).
 * ngp_pack_elites writes this rank's record: its n fitness values and its k best individuals, best first (ties: lower
 * index first).  ngp_unpack_elites reads the gathered records (rank order) and writes the global fitness vector
 * f64[sum n_r] and the sum k_r elites in rank order, ready to be passed to ngp_hof_update as a population: every rank
 * then holds the same hall of fame.  Any output may be NULL. */
int64_t ngp_exchange_bytes(const ngp_handle *h, int32_t n_max, int32_t k_max);
int ngp_pack_elites(ngp_handle *h, const float *genomes, const double *fitness, int32_t n, int32_t k, int32_t n_max,
                    int32_t k_max, void *out, void *stream);
int ngp_unpack_elites(ngp_handle *h, const void *gathered, int32_t world, int32_t n_max, int32_t k_max, double *fitness_all,
                      float *elite_genomes, double *elite_fitness, void *stream);

/* Tuning switches (experiments, geometry-independence tests): "rollout_block" (threads per CTA), "rollout_nosync",
 * "rollout_flavour" (1..3), "rollout_blocks_per_sm", "mlp_no_tf32", "select_os_min_t" (smallest tournament size that uses the
 * order-statistics selection, default 8192).  value 0 restores the automatic choice. */
int ngp_set_option(ngp_handle *h, const char *name, int64_t value);

/* Device-side timing of the dominant kernel (the fused rollout) with CUDA events recorded on the
 * launching stream around each launch.  ngp_profile_read synchronises the recorded events, returns
 * the accumulated milliseconds and launch count since the previous read, and resets both. */
int ngp_profile_enable(ngp_handle *h, int32_t on);
int ngp_profile_read(ngp_handle *h, double *rollout_ms, int32_t *rollout_launches);

/* kernels launched by this handle so far (bench.py's gpu_launches) */
uint64_t ngp_launch_count(const ngp_handle *h);

#ifdef __cplusplus
}
#endif
#endif
