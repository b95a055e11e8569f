// host_sim_matches.cpp -- TEST INFRASTRUCTURE: host_sim.cpp plus the match-list form of the fused rollout (ngp_play_matches),
// lanes executed one after another.  RolloutParams is filled as csrc/ngp_core.cu fills it for a match list: games = 1,
// match_right / match_left / match_mult set, scores written at the end of each episode as rollout_kernel writes them.
#include "host_sim.cpp"

extern "C" void hs_play_matches(void *h, int core, const int32_t *nodes, int n_layers, int bias, int max_frames, const float *genomes,
                                const int32_t *right, const int32_t *left, const double *mult, int n_matches, uint64_t seed,
                                uint64_t generation, double *rewards, int32_t *frames, int32_t *scores)
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
    a26::Ram ram{sim->ram_words};
    for (int e = 0; e < n_matches; ++e) {
        roll::Episode ep;
        a26::Chip s; a26::CpuRegs r;
        roll::episode_begin(ep, p, e, s, r, ram);
        double reward = 0.0;
        if (core) { while (!roll::episode_frame<1>(ep, p, s, r, sim->T, ram, &reward)) {} }
        else { while (!roll::episode_frame<0>(ep, p, s, r, sim->T, ram, &reward)) {} }
        p.rewards[e] = reward; p.frames[e] = ep.frame;
        p.scores[2 * e] = ep.last_s1; p.scores[2 * e + 1] = ep.last_s2;
    }
}
