// host_sim_states.cpp -- TEST INFRASTRUCTURE: host_sim.cpp plus ngp_play_matches_states, lanes executed one after another.
// The list check is match_check_kernel's (gs::match_entry_faults and gs::validate per start state); every match then runs as a
// lane of a recording twin of rollout_kernel does: episode_begin, resume_state, capture_state at capture_at[m], episode_frame
// <CORE, false, true>, record_frame when there is a record.
#include "host_sim.cpp"
#include "../../neuro_genetic_pong_self_play_b200/csrc/game_state.cuh"

extern "C" {

int hs_validate_state(const ngp_game_state *st, uint64_t cart) { return gs::validate(st, cart); }

// Returns the number of faults of the list check; with any, nothing is played and nothing is written.
long hs_play_states(void *h, int core, const int32_t *nodes, int n_layers, int bias, int max_frames, const float *genomes, int n_genomes,
                    const int32_t *right, const int32_t *left, const double *mult, const int32_t *key, int n_matches,
                    const ngp_game_state *states, int n_states, const int32_t *start, int fresh, const int32_t *capture_at,
                    ngp_game_state *capture, int max_record, ngp_frame_record *record, uint64_t cart, uint64_t seed, uint64_t generation,
                    double *rewards, int32_t *frames, int32_t *scores, uint64_t *frames_total)
{
    Sim *sim = (Sim *)h;
    long faults = 0;
    for (int m = 0; m < n_matches; ++m)
        faults += gs::match_entry_faults(m, right, left, n_genomes, key, capture_at, start, states, n_states);
    for (int k = 0; k < n_states; ++k) faults += gs::validate(states + k, cart) == 0;
    if (faults) return faults;
    roll::RolloutParams p;
    memset(&p, 0, sizeof(p));
    p.tables = &sim->T; p.needed = sim->needed.data(); p.start = sim->start;
    p.genomes = genomes;
    p.n = n_matches; p.games = 1; p.win_score = 3; p.timeout_thresh = 2000; p.max_frames = max_frames;
    p.core = core; p.time_scaler = 100.0; p.paddle_height = 16.0; p.seed = seed; p.generation = generation;
    p.shape.n_layers = n_layers; p.shape.bias = bias;
    int G = 0;
    for (int i = 0; i < n_layers; ++i) p.shape.nodes[i] = nodes[i];
    for (int i = 0; i + 1 < n_layers; ++i) G += (nodes[i] + (bias ? 1 : 0)) * nodes[i + 1];
    p.G = G;
    p.match_right = right; p.match_left = left; p.match_mult = mult;
    p.rewards = rewards; p.frames = frames; p.scores = scores;
    for (int players = 1; players <= 2; ++players)
        for (int la = 0; la < 3; ++la)
            for (int ra = 0; ra < 3; ++ra) {
                uint8_t a[16] = {0};
                a[0] = 1; a[15] = 1;
                a[4] = ra == pol::ACT_UP; a[5] = ra == pol::ACT_DOWN;
                a[6] = la == pol::ACT_UP; a[7] = la == pol::ACT_DOWN;
                p.input_table[players - 1][la * 3 + ra] = roll::action_to_input(a, players, kDefaultButtonMap);
            }
    roll::RecordArgs rec;
    memset(&rec, 0, sizeof(rec));
    rec.record = record; rec.key = key; rec.max_record = record ? max_record : 0;
    rec.fresh = fresh; rec.states = states; rec.start = start; rec.capture_at = capture_at; rec.capture = capture; rec.cart = cart;
    a26::Ram ram{sim->ram_words};
    uint64_t total = 0;
    for (int e = 0; e < n_matches; ++e) {
        roll::Episode ep;
        a26::Chip s; a26::CpuRegs r;
        roll::episode_begin(ep, p, e, s, r, ram);
        if (rec.start && rec.start[e] >= 0) roll::resume_state(rec, rec.start[e], ep, s, r, ram);
        const int capture_frame = rec.capture_at ? rec.capture_at[e] : -1;
        if (capture_frame == ep.frame) roll::capture_state(rec, ep, s, r, ram);
        double reward = 0.0;
        for (;;) {
            const bool done = core ? roll::episode_frame<1, false, true>(ep, p, s, r, sim->T, ram, &reward, true, &rec)
                                   : roll::episode_frame<0, false, true>(ep, p, s, r, sim->T, ram, &reward, true, &rec);
            ++total;
            if (rec.record && ep.frame <= rec.max_record) roll::record_frame(rec, ep, s, ep.last_s1, ep.last_s2);
            if (!done && ep.frame == capture_frame) roll::capture_state(rec, ep, s, r, ram);
            if (done) break;
        }
        p.rewards[e] = reward; p.frames[e] = ep.frame;
        p.scores[2 * e] = ep.last_s1; p.scores[2 * e + 1] = ep.last_s2;
    }
    *frames_total = total;
    return 0;
}

}  // extern "C"
