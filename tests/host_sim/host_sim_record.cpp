// host_sim_record.cpp -- TEST INFRASTRUCTURE: host_sim.cpp plus the recording form of the fused rollout
// (ngp_record_matches), lanes executed one after another.  RolloutParams is filled as for a match list (host_sim_matches.cpp);
// every frame runs episode_frame<CORE, false, true> and then record_frame, as the recording twins of rollout_kernel do.
#include "host_sim.cpp"

extern "C" void hs_record_matches(void *h, int core, const int32_t *nodes, int n_layers, int bias, int max_frames, const float *genomes,
                                  const int32_t *right, const int32_t *left, const double *mult, const int32_t *key, int n_matches,
                                  uint64_t seed, uint64_t generation, int max_record, ngp_frame_record *record, double *rewards,
                                  int32_t *frames, int32_t *scores)
{
    Sim *sim = (Sim *)h;
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
    rec.record = record; rec.key = key; rec.max_record = max_record;
    a26::Ram ram{sim->ram_words};
    for (int e = 0; e < n_matches; ++e) {
        roll::Episode ep;
        a26::Chip s; a26::CpuRegs r;
        roll::episode_begin(ep, p, e, s, r, ram);
        double reward = 0.0;
        for (;;) {
            const bool done = core ? roll::episode_frame<1, false, true>(ep, p, s, r, sim->T, ram, &reward, true, &rec)
                                   : roll::episode_frame<0, false, true>(ep, p, s, r, sim->T, ram, &reward, true, &rec);
            if (ep.frame <= rec.max_record) roll::record_frame(rec, ep, s, ep.last_s1, ep.last_s2);
            if (done) break;
        }
        p.rewards[e] = reward; p.frames[e] = ep.frame;
        p.scores[2 * e] = ep.last_s1; p.scores[2 * e + 1] = ep.last_s2;
    }
}

// hs_create with other target colours of find_stuff (ngp_config.ball_colour / left_colour / right_colour): a colour that
// matches nothing hides that object from the observation, e.g. to force get_actions' random fall-back.
extern "C" void *hs_create_colours(const uint8_t *rom, const uint8_t *ball, const uint8_t *left, const uint8_t *right)
{
    Sim *sim = new Sim();
    ngp_host::build_tables(sim->T, rom, ball, left, right, kPalette);
    sim->needed.resize(a26::TRIGMAX + 1);
    ngp_host::build_paddle_table(sim->needed.data());
    a26::Ram ram{sim->ram_words};
    for (int st = 0; st < 2; ++st) {
        roll::build_start_state(st, sim->s, sim->r, sim->T, ram, sim->needed.data());
        roll::store_snapshot(&sim->start[st], sim->s, sim->r, ram);
    }
    return sim;
}
