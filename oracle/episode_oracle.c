/* episode_oracle.c -- CPU ORACLE (test infrastructure, NOT product code).  See episode_oracle.h
 * for the reference file:line each function follows.  Compile with -ffp-contract=off: the
 * double arithmetic here is meant to be reproduced bit-for-bit by the CUDA core. */
#include "episode_oracle.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>

/* config.py:3-6 */
static const uint8_t TARGET_COLOURS[3][3] = {{236, 236, 236}, {213, 130, 74}, {92, 186, 92}};

/* ---------------------------------------------------------------- utils.py:128-136 ---- */
int eo_gene_size(const eo_shape *sh)
{
    int total = 0;
    for (int i = 0; i + 1 < sh->n_layers; ++i) total += (sh->nodes[i] + (sh->bias ? 1 : 0)) * sh->nodes[i + 1];
    return total;
}

/* Deterministic exp: only IEEE-754 double +,*,floor and bit assembly, so the CUDA core can
 * reproduce it bit-for-bit.  |rel err| < 3e-16 on the sigmoid's input range. */
double eo_det_exp(double x)
{
    static const double LN2_HI = 6.93147180369123816490e-01, LN2_LO = 1.90821492927058770002e-10,
                        INV_LN2 = 1.44269504088896338700e+00;
    if (x != x) return x;
    if (x > 709.0) return INFINITY;
    if (x < -708.0) return 0.0;
    double k = floor(x * INV_LN2 + 0.5);
    double r = (x - k * LN2_HI) - k * LN2_LO;
    /* Taylor to r^13 on |r| <= 0.3466, Horner */
    double p = 1.0 / 6227020800.0;
    p = p * r + 1.0 / 479001600.0;
    p = p * r + 1.0 / 39916800.0;
    p = p * r + 1.0 / 3628800.0;
    p = p * r + 1.0 / 362880.0;
    p = p * r + 1.0 / 40320.0;
    p = p * r + 1.0 / 5040.0;
    p = p * r + 1.0 / 720.0;
    p = p * r + 1.0 / 120.0;
    p = p * r + 1.0 / 24.0;
    p = p * r + 1.0 / 6.0;
    p = p * r + 0.5;
    p = p * r + 1.0;
    p = p * r + 1.0;
    int64_t ki = (int64_t)k;
    uint64_t bits = (uint64_t)(ki + 1023) << 52;
    double scale;
    memcpy(&scale, &bits, 8);
    return p * scale;
}

/* ------------------------------------------------------ numpy_nn.py:35-69, 120-137 ---- */
void eo_mlp_forward(const eo_shape *sh, const float *genome, const double *x, double *out, int *action)
{
    double buf_a[4097], buf_b[4097];                  /* layers up to 4096 units plus the bias input */
    double *cur = buf_a, *nxt = buf_b;
    int n_in = sh->nodes[0];
    int bias = sh->bias ? 1 : 0;
    for (int i = 0; i < n_in; ++i) cur[i] = x[i];
    const float *w = genome;
    for (int l = 0; l + 1 < sh->n_layers; ++l) {
        int ni = sh->nodes[l], no = sh->nodes[l + 1];
        if (bias) cur[ni] = 1.0;                      /* trailing bias input, weight = LAST column */
        for (int o = 0; o < no; ++o) {
            double z = 0.0;
            for (int i = 0; i < ni + bias; ++i) z = z + (double)w[o * (ni + bias) + i] * cur[i];
            nxt[o] = 1.0 / (1.0 + eo_det_exp(-z));    /* sigmoid on every layer incl. output */
        }
        w += (ni + bias) * no;
        double *t = cur; cur = nxt; nxt = t;
    }
    int n_out = sh->nodes[sh->n_layers - 1];
    int best = 0;
    for (int o = 0; o < n_out; ++o) {
        if (out) out[o] = cur[o];
        if (cur[o] > cur[best]) best = o;             /* np.argmax: first maximum wins */
    }
    if (action) *action = best == 0 ? EO_ACT_UP : EO_ACT_DOWN;
}

/* ----------------------------------------------------------- utils.py:14-19, 60-68 ---- */
void eo_find_stuff(const uint8_t *rgb, eo_obs *out)
{
    for (int t = 0; t < 3; ++t) {
        int64_t cnt = 0, sr = 0, sc = 0;
        for (int r = EO_GAME_TOP; r < EO_GAME_BOTTOM; ++r)
            for (int c = 0; c < 160; ++c)
                for (int ch = 0; ch < 3; ++ch)        /* per-CHANNEL matches, as argwhere(chopped == colour) */
                    if (rgb[(r * 160 + c) * 3 + ch] == TARGET_COLOURS[t][ch]) {
                        cnt++; sr += r - EO_GAME_TOP; sc += c;
                    }
        out->valid[t] = cnt > 0;
        out->loc[t][0] = cnt ? (double)sr / (double)cnt : 0.0;
        out->loc[t][1] = cnt ? (double)sc / (double)cnt : 0.0;
    }
}

/* ---------------------------------------------------------------- utils.py:71-77 ------ */
int eo_clamp(int valid, double paddle_row, int action)
{
    if (valid) {
        if (paddle_row < EO_PADDLE_HEIGHT) return EO_ACT_DOWN;
        else if (paddle_row > (EO_GAME_BOTTOM - EO_GAME_TOP) - EO_PADDLE_HEIGHT) return EO_ACT_UP;
    }
    return action;
}

/* ---------------------------------------------------------------- utils.py:104-109 ---- */
double eo_reward(double mult, double total_frames, int my_score, int enemy_score)
{
    double diff = (double)(my_score - enemy_score);
    double scaled_time = total_frames / EO_TIME_SCALER;
    double bonus = (double)my_score * mult;
    return (diff + bonus) / scaled_time;
}

/* ------------------------------------------------------------------ Philox4x32-10 ----- */
void eo_philox4x32(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

/* the reference's np.random.choice(2) per player per frame (utils.py:112-113, main.py:139-140),
 * made reproducible: counter = (env, frame, 2*generation + player, 'PONG'), key = seed */
uint32_t eo_philox_bit(uint64_t seed, uint64_t generation, uint32_t env_id, uint32_t frame, uint32_t stream)
{
    uint32_t ctr[4] = {env_id, frame, ((uint32_t)generation << 1) | stream, 0x504F4E47u}, key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)}, out[4];
    eo_philox4x32(ctr, key, out);
    return out[0] & 1u;
}

/* -------------------------------------------------------- config.py:15-23, main.py:91-92 */
/* gym-retro's button vector -> console input.  [3P-recall] 8 buttons per player (BUTTON, -, SELECT, RESET, UP, DOWN, LEFT,
 * RIGHT); an env made with players=1 (main.py:40) consumes only action[0:8]; FILTERED cancels UP+DOWN / LEFT+RIGHT of one
 * player.  What each button does to the console is a table (EO_BTN_*), by default the reference's own names: [0]
 * RIGHT_PLAYER_START_BUTTON = fire of paddle 1, [15] LEFT_PLAYER_START_BUTTON = fire of paddle 0, [4]/[5] = right player
 * (paddle 1) up/down, [6]/[7] = left player (paddle 0) up/down.  "up" (the reference's [1,0]) = lower resistance. */
static uint8_t g_button_map[16] = {EO_BTN_FIRE_P0 + 1, 0, EO_BTN_SELECT, EO_BTN_RESET, EO_BTN_UP_P0 + 2, EO_BTN_UP_P0 + 3,
                                   EO_BTN_UP_P0 + 0, EO_BTN_UP_P0 + 1, 0, 0, EO_BTN_SELECT, EO_BTN_RESET, 0, 0, 0, EO_BTN_FIRE_P0 + 0};
void eo_set_button_map(const uint8_t map[16]) { memcpy(g_button_map, map, 16); }
void eo_get_button_map(uint8_t map[16]) { memcpy(map, g_button_map, 16); }

void eo_action_to_input(const uint8_t action[16], int players, a26o_input *in)
{
    in->swchb = 0x3F; in->fire = 0; in->dec = 0; in->inc = 0;
    for (int p = 0; p < players && p < 2; ++p) {
        const uint8_t *b = action + 8 * p;
        const uint8_t *m = g_button_map + 8 * p;
        int held[8];
        for (int i = 0; i < 8; ++i) held[i] = b[i] != 0;
        if (held[4] && held[5]) held[4] = held[5] = 0;      /* retro.Actions.FILTERED */
        if (held[6] && held[7]) held[6] = held[7] = 0;
        for (int i = 0; i < 8; ++i) {
            if (!held[i]) continue;
            int code = m[i];
            if (code >= EO_BTN_FIRE_P0 && code < EO_BTN_FIRE_P0 + 4) in->fire |= (uint8_t)(1 << (code - EO_BTN_FIRE_P0));
            else if (code >= EO_BTN_UP_P0 && code < EO_BTN_UP_P0 + 8) {
                int paddle = (code - EO_BTN_UP_P0) / 2;
                if ((code - EO_BTN_UP_P0) % 2) in->inc |= (uint8_t)(1 << paddle); else in->dec |= (uint8_t)(1 << paddle);
            } else if (code == EO_BTN_SELECT) in->swchb &= (uint8_t)~0x02;
            else if (code == EO_BTN_RESET) in->swchb &= (uint8_t)~0x01;
        }
    }
}

static void idle(a26o *env, uint8_t swchb, int frames)
{
    a26o_input in = {swchb, 0, 0, 0};
    for (int i = 0; i < frames; ++i) a26o_run_frame(env, &in, NULL);
}

void eo_reset_to_state(a26o *env, int state_id)
{
    a26o_power_on(env);
    idle(env, 0x3F, 8);
    if (state_id == EO_STATE_START_2P) {            /* SELECT twice: game 1 -> game 3 (2-player Pong) */
        idle(env, 0x3F & ~0x02, 1); idle(env, 0x3F, 1);
        idle(env, 0x3F & ~0x02, 1); idle(env, 0x3F, 1);
    }
    idle(env, 0x3F & ~0x01, 2);                      /* RESET */
    idle(env, 0x3F, 1);                              /* <- the save state */
    idle(env, 0x3F, 1);                              /* gym-retro reset(): one frame, no buttons */
}

/* ---------------------------------------------------------------- dumb_ais.py ---------- */
static int hardcoded(const double x[6])
{
    if (x[1] < x[4]) return EO_ACT_UP;
    if (x[1] > x[4]) return EO_ACT_DOWN;
    return EO_ACT_NONE;
}

/* dumb_ais.py:1-8 (kind EO_POLICY_HARDCODED) and :11-25 (EO_POLICY_SCORE_HARDCODED, after set_score) */
int eo_bot_act(int kind, const double x[6], int score1, int score2)
{
    if (kind == EO_POLICY_SCORE_HARDCODED && !(score1 <= score2)) return EO_ACT_NONE;
    return hardcoded(x);
}

/* utils.py:139-153: the six-vector handed to model.run */
void eo_inference_vector(const double ball[2], const double last[2], double me_row, double enemy_row, double x[6])
{
    x[0] = ball[1] / EO_GAME_WIDTH; x[1] = ball[0] / EO_PLAYABLE_HEIGHT; x[2] = last[1] / EO_GAME_WIDTH;
    x[3] = last[0] / EO_PLAYABLE_HEIGHT; x[4] = me_row / EO_PLAYABLE_HEIGHT; x[5] = enemy_row / EO_PLAYABLE_HEIGHT;
}

/* utils.py:139-153 + model.run */
static int inference(const eo_shape *sh, const double ball[2], const double last[2], double me_row, double enemy_row,
                     eo_policy pol, int score1, int score2)
{
    double x[6];
    int act;
    eo_inference_vector(ball, last, me_row, enemy_row, x);
    switch (pol.kind) {
    case EO_POLICY_HARDCODED:
    case EO_POLICY_SCORE_HARDCODED: return eo_bot_act(pol.kind, x, score1, score2);
    default: eo_mlp_forward(sh, pol.genome, x, NULL, &act); return act;
    }
}

/* ---------------------------------------------------------------- main.py:69-112 ------- */
void eo_episode(a26o *env, const eo_shape *shape, eo_policy left, eo_policy right, double mult,
                uint64_t seed, uint64_t generation, uint32_t env_id, int players, int max_frames, eo_episode_result *res,
                uint8_t *trace, int trace_cap)
{
    uint8_t action[16] = {0};
    uint8_t fb[A26O_FB_ROWS * A26O_FB_COLS];
    uint8_t *rgb = (uint8_t *)malloc(A26O_FB_ROWS * A26O_FB_COLS * 3);
    action[0] = 1; action[15] = 1;                    /* BLANK_ACTION, config.py:21-23 */
    int have_last_score = 0, last_s1 = 0, last_s2 = 0;
    double timeout = 0.0, total_frames = 0.0;
    int have_last_ball = 0;
    double last_ball[2] = {0, 0};
    int frame = 0, s1 = 0, s2 = 0;
    for (;;) {
        a26o_input in;
        eo_action_to_input(action, players, &in);
        a26o_run_frame(env, &in, fb);
        a26o_fb_to_rgb(fb, rgb);
        s1 = a26o_ram(env)[13]; s2 = a26o_ram(env)[14];
        eo_obs ob;
        eo_find_stuff(rgb, &ob);
        /* main.get_actions (main.py:138-154) */
        int left_act = eo_philox_bit(seed, generation, env_id, (uint32_t)frame, 0) ? EO_ACT_DOWN : EO_ACT_UP;
        int right_act = eo_philox_bit(seed, generation, env_id, (uint32_t)frame, 1) ? EO_ACT_DOWN : EO_ACT_UP;
        if (ob.valid[0]) {
            const double *ball = ob.loc[0];
            double lb[2] = {have_last_ball ? last_ball[0] : ball[0], have_last_ball ? last_ball[1] : ball[1]};
            /* deviation (SURVEY Appendix A5): the reference raises TypeError when the enemy paddle is
             * missing; here the random action is kept in that case */
            if (ob.valid[1] && ob.valid[2]) {
                double fball[2] = {ball[0], EO_GAME_WIDTH - ball[1]}, flast[2] = {lb[0], EO_GAME_WIDTH - lb[1]};
                left_act = inference(shape, fball, flast, ob.loc[1][0], ob.loc[2][0], left, s1, s2);
                right_act = inference(shape, ball, lb, ob.loc[2][0], ob.loc[1][0], right, s1, s2);
            }
        } else {
            left_act = EO_ACT_NONE; right_act = EO_ACT_NONE;
        }
        have_last_ball = ob.valid[0];
        if (ob.valid[0]) { last_ball[0] = ob.loc[0][0]; last_ball[1] = ob.loc[0][1]; }
        left_act = eo_clamp(ob.valid[1], ob.loc[1][0], left_act);
        right_act = eo_clamp(ob.valid[2], ob.loc[2][0], right_act);
        action[4] = right_act == EO_ACT_UP; action[5] = right_act == EO_ACT_DOWN;
        action[6] = left_act == EO_ACT_UP;  action[7] = left_act == EO_ACT_DOWN;
        /* main.calculate_timeout_and_frames (main.py:128-135) */
        if (have_last_score) {
            if (last_s1 == s1 && last_s2 == s2) timeout += 1.0;
            else { total_frames += timeout; timeout = 0.0; }
        }
        have_last_score = 1; last_s1 = s1; last_s2 = s2;
        if (trace && frame < trace_cap) {
            uint8_t *t = trace + (size_t)frame * 144;
            memcpy(t, a26o_ram(env), 128);
            t[128] = (uint8_t)left_act; t[129] = (uint8_t)right_act; t[130] = (uint8_t)s1; t[131] = (uint8_t)s2;
            t[132] = ob.valid[0]; t[133] = ob.valid[1]; t[134] = ob.valid[2]; t[135] = 0;
            uint32_t to = (uint32_t)timeout, fr = (uint32_t)frame;
            memcpy(t + 136, &to, 4); memcpy(t + 140, &fr, 4);
        }
        frame++;
        if (s1 >= EO_WIN_SCORE || s2 >= EO_WIN_SCORE) break;
        if (timeout > EO_TIMEOUT_THRESH) break;
        if (max_frames > 0 && frame >= max_frames) break;
    }
    res->frames = frame; res->score1 = s1; res->score2 = s2; res->total_frames = total_frames;
    res->reward = s1 == s2 ? 0.0 : eo_reward(mult, total_frames, s2, s1);
    free(rgb);
}

/* ---------------------------------------------------------------- main.py:28-66 -------- */
double eo_evaluate(const uint8_t rom[2048], const eo_shape *shape, const float *genome,
                   const float *hof_genomes, const double *hof_fitness, int n_hof, const int hof_pick[3],
                   uint64_t seed, uint64_t generation, uint32_t genome_id, double rewards[EO_GAMES_TO_PLAY], int frames[EO_GAMES_TO_PLAY])
{
    a26o *env = a26o_new(rom);
    int G = eo_gene_size(shape);
    double mult = 1.0, sum = 0.0;
    eo_policy right = {EO_POLICY_MLP, genome};
    for (int i = 0; i < EO_GAMES_TO_PLAY; ++i) {
        eo_policy left = {EO_POLICY_HARDCODED, NULL};
        int state = EO_STATE_START_2P;
        if (i == 1) state = EO_STATE_START_1P;
        else if (i == 2) left.kind = EO_POLICY_SCORE_HARDCODED;
        else if (i >= 3) {
            mult = 1.0;                               /* utils.py:92: reset to 1 on every call */
            if (n_hof > 0) {
                int h = hof_pick[i - 3];
                mult = hof_fitness[h];
                left.kind = EO_POLICY_MLP; left.genome = hof_genomes + (size_t)h * G;
            }
        }
        eo_reset_to_state(env, state);
        eo_episode_result r;
        eo_episode(env, shape, left, right, mult, seed, generation, genome_id * EO_GAMES_TO_PLAY + (uint32_t)i,
                   state == EO_STATE_START_1P ? 1 : 2, 0, &r, NULL, 0);
        rewards[i] = r.reward; frames[i] = r.frames;
        sum += r.reward;
    }
    a26o_free(env);
    return sum / (double)EO_GAMES_TO_PLAY;
}

void eo_selfplay_game(const uint8_t rom[2048], const eo_shape *shape, const float *right, const float *left,
                      uint64_t seed, uint64_t generation, uint32_t env_id, eo_episode_result *res)
{
    a26o *env = a26o_new(rom);
    eo_policy l = {EO_POLICY_MLP, left}, r = {EO_POLICY_MLP, right};
    eo_reset_to_state(env, EO_STATE_START_2P);
    eo_episode(env, shape, l, r, 1.0, seed, generation, env_id, 2, 0, res, NULL, 0);
    a26o_free(env);
}
