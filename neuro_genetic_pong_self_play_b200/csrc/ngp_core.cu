// ngp_core.cu -- handle management, the batched 2600 core kernels (K1) and the fused
// population-evaluation rollout (K1+K2+K3 + episode control) of libngp.so.
//
// Reference path replaced (file:line in the reference tree):
//   main.evaluate 28-66, main.perform_episode 69-112, main.get_actions 138-154,
//   main.calculate_timeout_and_frames 128-135, utils.find_stuff 14-19/60-68, utils.inference
//   139-153, numpy_nn.NeuralNetwork.run 120-137, dumb_ais 1-25, utils.keep_within_game_bounds_please
//   71-77, utils.calculate_reward 104-109, and gym-retro's env.reset/env.step underneath.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <memory>
#include <mutex>
#include <vector>

#include "ngp_internal.h"
#include "rollout_kernel.cuh"
#include "host_tables.h"

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
void ngp_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
extern "C" const char *ngp_last_error(void) { return g_err; }
extern "C" const char *ngp_version(void) { return "ngp 0.1 (sm_100a)"; }

extern "C" void ngp_default_config(ngp_config *cfg, int32_t population)
{
    memset(cfg, 0, sizeof(*cfg));
    cfg->n_layers = 3;
    cfg->nodes[0] = 6; cfg->nodes[1] = 2; cfg->nodes[2] = 2;        // NETWORK_SHAPE
    cfg->bias = 1;
    cfg->games_to_play = NGP_GAMES_TO_PLAY;
    cfg->win_score = 3;
    cfg->timeout_thresh = 2000;
    cfg->schedule = NGP_SCHEDULE_REFERENCE;
    cfg->max_frames = 0;
    cfg->time_scaler = 100.0f;
    cfg->scaled_paddle_height = 16.0f;
    const uint8_t ball[3] = {236, 236, 236}, left[3] = {213, 130, 74}, right[3] = {92, 186, 92};
    memcpy(cfg->ball_colour, ball, 3); memcpy(cfg->left_colour, left, 3); memcpy(cfg->right_colour, right, 3);
    cfg->cxpb = 0.9f; cfg->cx_alpha = 0.9f; cfg->mutpb = 0.9f; cfg->mut_mu = 0.0f; cfg->mut_sigma = 0.9f; cfg->mut_indpb = 0.9f;
    cfg->tournament_size = population / 4;
    cfg->core = NGP_CORE_TRANSLATED;
    ngp_host::default_button_map(cfg->button_map);
}

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
using a26::Chip; using a26::CpuRegs; using a26::Ram; using a26::Snapshot; using a26::Tables;
using roll::RolloutParams; using roll::load_snapshot; using roll::store_snapshot; using roll::action_to_input;
using pol::ACT_UP; using pol::ACT_DOWN;

// ------------------------------------------------------------------------------------------------
// start-state construction: power-on + scripted console switches (DESIGN.md "start states")
// ------------------------------------------------------------------------------------------------
__global__ void build_start_states_kernel(const Tables *tables, const uint32_t *needed, Snapshot *out)
{
    __shared__ Tables T;
    __shared__ uint32_t ram_smem[32 * 32];
    load_tables(T, tables);
    const int state = blockIdx.x;                 // one CTA (one lane of it) per start state: the two scripts diverge from the first frame
    if (threadIdx.x != 0 || state >= 2) return;
    Ram ram{&ram_smem[threadIdx.x]};
    Chip s; CpuRegs r;
    roll::build_start_state(state, s, r, T, ram, needed);
    store_snapshot(&out[state], s, r, ram);
}

// ------------------------------------------------------------------------------------------------
// K1 stepwise (verify mode)
// ------------------------------------------------------------------------------------------------
__global__ void env_reset_kernel(const Snapshot *start, Snapshot *envs, int n)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) envs[i] = *start;
}

struct ButtonMap { uint8_t m[16]; };

template <bool VERIFY>
__global__ void __launch_bounds__(32) env_step_kernel(const Tables *tables, const uint32_t *needed, Snapshot *envs, int n, int lanes, int core, int players, ButtonMap map,
                                                      const uint8_t *actions, uint8_t *fb, uint8_t *ram_out, float *loc,
                                                      uint8_t *valid, uint8_t *regs, unsigned long long *counters)
{
    __shared__ Tables T;
    __shared__ uint32_t ram_smem[32 * 32];
    load_tables(T, tables);
    // `lanes` environments per warp: a small batch is spread over the SMs (stepwise environments follow unrelated action
    // traces, so the lanes of a warp mostly take turns; one environment per warp runs them side by side)
    const int e = blockIdx.x * lanes + threadIdx.x;
    if ((int)threadIdx.x >= lanes || e >= n) return;
    Ram ram{&ram_smem[threadIdx.x]};
    Chip s; CpuRegs r;
    load_snapshot(&envs[e], s, r, ram);
    const uint32_t in = action_to_input(actions + (size_t)e * 16, players, map.m);
    a26::apply_input(s, needed, in & 0xFF, (in >> 8) & 15, (in >> 12) & 15, (in >> 16) & 15);
    a26::clear_obs(s);
    uint8_t *my_fb = fb ? fb + (size_t)e * a26::FB_ROWS * a26::FB_COLS : nullptr;
    if (core) a26::run_frame_compiled<VERIFY, false>(s, r, T, ram, my_fb);
    else a26::run_frame<VERIFY>(s, r, T, ram, my_fb);
    store_snapshot(&envs[e], s, r, ram);
    if (s.error) atomicAdd(&counters[2], 1ull);
    if (ram_out) for (int i = 0; i < 128; ++i) ram_out[(size_t)e * 128 + i] = (uint8_t)ram.rd(i);
    if (loc && valid)
        for (int t = 0; t < 3; ++t) {
            valid[e * 3 + t] = s.cnt[t] > 0;
            loc[(e * 3 + t) * 2 + 0] = s.cnt[t] ? (float)__ddiv_rn((double)s.sy[t], (double)s.cnt[t]) : 0.f;
            loc[(e * 3 + t) * 2 + 1] = s.cnt[t] ? (float)__ddiv_rn((double)s.sx[t], (double)s.cnt[t]) : 0.f;
        }
    if (regs) {
        uint8_t *o = regs + (size_t)e * 8;
        o[0] = (uint8_t)r.a; o[1] = (uint8_t)r.x; o[2] = (uint8_t)r.y; o[3] = (uint8_t)r.sp; o[4] = (uint8_t)a26::pack_p(r);
        o[5] = (uint8_t)r.pc; o[6] = (uint8_t)(r.pc >> 8); o[7] = s.error;
    }
}

__global__ void palette_to_rgb_kernel(const uint8_t *__restrict__ fb, const uint32_t *__restrict__ palette, uint8_t *__restrict__ rgb, size_t n_pixels)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pixels) return;
    uint32_t c = palette[fb[i] >> 1];
    rgb[3 * i + 0] = (uint8_t)(c >> 16); rgb[3 * i + 1] = (uint8_t)(c >> 8); rgb[3 * i + 2] = (uint8_t)c;
}

__global__ void env_digest_kernel(const Snapshot *envs, int n, uint32_t *out)
{
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const Chip &s = envs[e].chip;
    uint32_t *o = out + (size_t)e * 8;
    o[0] = s.cx;
    o[1] = (uint32_t)s.posp0 | ((uint32_t)s.posp1 << 8) | ((uint32_t)s.posm0 << 16) | ((uint32_t)s.posm1 << 24);
    o[2] = (uint32_t)s.posbl | ((uint32_t)s.vblank << 8) | ((uint32_t)s.ctrlpf << 16) | ((uint32_t)s.vdelbl << 24);
    o[3] = (uint32_t)s.charge[0] | ((uint32_t)s.charge[1] << 16);
    o[4] = (uint32_t)s.charge[2] | ((uint32_t)s.charge[3] << 16);
    o[5] = (uint32_t)s.grp0_new | ((uint32_t)s.grp1_new << 8) | ((uint32_t)s.enabl_new << 16) | ((uint32_t)s.enabl_old << 24);
    o[6] = (envs[e].cpu.cyc - envs[e].cpu.cpu_ls) % a26::LINE_CYCLES;
    o[7] = s.dump_enabled;
}

int ngp_evaluate_stepwise(ngp_handle *h, const RolloutParams &p, cudaStream_t st);     // ngp_stepwise.cu

// fitness[g] = sum(rewards[g][:]) / games, summed in game order (main.py:65)
__global__ void fitness_reduce_kernel(const double *__restrict__ rewards, int n, int games, double *__restrict__ fitness)
{
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n) return;
    double sum = 0.0;
    for (int k = 0; k < games; ++k) sum = __dadd_rn(sum, rewards[(size_t)g * games + k]);
    fitness[g] = __ddiv_rn(sum, (double)games);
}

// the argument check of the match-list entry points: counts the faults of every match entry (gs::match_entry_faults) and the
// start states that fail validation
__global__ void match_check_kernel(const int32_t *__restrict__ right, const int32_t *__restrict__ left, const int32_t *__restrict__ key,
                                   int n, int n_genomes, const int32_t *__restrict__ capture_at, const int32_t *__restrict__ start,
                                   const ngp_game_state *__restrict__ states, int n_states, uint64_t cart, unsigned long long *bad)
{
    unsigned long long c = 0;
    for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < n; m += gridDim.x * blockDim.x)
        c += gs::match_entry_faults(m, right, left, n_genomes, key, capture_at, start, states, n_states);
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_states; k += gridDim.x * blockDim.x) c += gs::validate(states + k, cart) == 0;
    if (c) atomicAdd(bad, c);
}

// stepwise save states: pack every environment (no episode) / count the bad states of a set and, in bad[1], take the players
// value of the first / unpack them into the environments
__global__ void env_get_state_kernel(Snapshot *envs, int n, int players, uint64_t cart, ngp_game_state *out)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n) gs::pack(out + e, cart, players, envs[e].chip, envs[e].cpu, gs::SnapRam{envs[e].ram}, nullptr);
}
__global__ void state_check_kernel(const ngp_game_state *states, int n, uint64_t cart, unsigned long long *bad)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const int players = gs::validate(states + e, cart), first = gs::validate(states, cart);
    if (players == 0 || players != first) atomicAdd(bad, 1ull);
    if (e == 0) bad[1] = (unsigned long long)players;
}
__global__ void env_set_state_kernel(const ngp_game_state *states, Snapshot *envs, int n)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n) gs::unpack(states + e, envs[e].chip, envs[e].cpu, gs::SnapRam{envs[e].ram}, nullptr);
}

// ------------------------------------------------------------------------------------------------
// host API
// ------------------------------------------------------------------------------------------------
extern "C" int32_t ngp_gene_size(const ngp_handle *h) { return h ? h->gene_size : 0; }
extern "C" uint64_t ngp_launch_count(const ngp_handle *h) { return h ? h->launches : 0; }

static std::mutex g_start_mutex;
static std::map<uint64_t, std::vector<Snapshot>> g_start_cache;       // cartridge hash -> {'Start', 'Start.2P'} (immutable)
static uint64_t fnv1a64(const uint8_t *p, size_t n)
{
    uint64_t hsh = 1469598103934665603ull;
    for (size_t i = 0; i < n; ++i) { hsh ^= p[i]; hsh *= 1099511628211ull; }
    return hsh;
}

extern "C" int32_t ngp_config_size(void) { return (int32_t)sizeof(ngp_config); }

// Tuning switches that used to be environment variables; 0 restores the automatic choice.
extern "C" int ngp_set_option(ngp_handle *h, const char *name, int64_t value)
{
    NGP_REQUIRE(h && name, "ngp_set_option: bad arguments");
    const std::string n(name);
    if (n == "rollout_block") h->opt_rollout_block = (int)value;
    else if (n == "rollout_nosync") h->opt_rollout_nosync = value != 0;
    else if (n == "rollout_flavour") h->opt_rollout_lean = (int)value;
    else if (n == "rollout_blocks_per_sm") h->opt_rollout_blocks_per_sm = (int)value;
    else if (n == "mlp_no_tf32") h->opt_mlp_no_tf32 = value != 0;
    else if (n == "select_os_min_t") h->opt_select_os_min_t = (int)value;
    else { ngp_set_error("ngp_set_option: unknown option '%s'", name); return NGP_ERR_INVALID; }
    return NGP_OK;
}

extern "C" int ngp_create(const ngp_config *cfg, const uint8_t *rom, int32_t device, ngp_handle **out)
{
    NGP_REQUIRE(cfg && rom && out, "ngp_create: null argument");
    NGP_REQUIRE(cfg->n_layers >= 2 && cfg->n_layers <= NGP_MAX_LAYERS, "ngp_create: n_layers out of range");
    NGP_REQUIRE(cfg->nodes[0] == 6, "ngp_create: the observation vector has 6 entries (utils.py:139-153)");
    NGP_REQUIRE(cfg->games_to_play >= 1 && cfg->games_to_play <= 64, "ngp_create: games_to_play out of range");
    int count = 0;
    NGP_CUDA(cudaGetDeviceCount(&count));
    NGP_REQUIRE(device >= 0 && device < count, "ngp_create: no such CUDA device");
    NGP_CUDA(cudaSetDevice(device));
    auto h = std::make_unique<ngp_handle>();     // freed with everything it holds on an early return
    h->cfg = *cfg;
    h->device = device;
    h->shape.n_layers = cfg->n_layers;
    for (int i = 0; i < 8; ++i) h->shape.nodes[i] = cfg->nodes[i];
    h->shape.bias = cfg->bias;
    h->gene_size = pol::gene_size(h->shape);
    NGP_CUDA(cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device));

    h->rom_translated = a26::rom_matches_translation(rom) ? 1 : 0;
    h->cart_hash = fnv1a64(rom, 2048);
    Tables tables;
    ngp_host::build_tables(tables, rom, cfg->ball_colour, cfg->left_colour, cfg->right_colour, ngp_host::ntsc_palette);
    std::vector<uint32_t> needed(a26::TRIGMAX + 1);
    ngp_host::build_paddle_table(needed.data());
    NGP_CUDA(h->d_tables.ensure(1));
    NGP_CUDA(cudaMemcpy(h->d_tables.p, &tables, sizeof(Tables), cudaMemcpyHostToDevice));
    NGP_CUDA(h->d_needed.ensure(needed.size()));
    NGP_CUDA(cudaMemcpy(h->d_needed.p, needed.data(), needed.size() * 4, cudaMemcpyHostToDevice));
    NGP_CUDA(h->d_palette.ensure(128));
    NGP_CUDA(cudaMemcpy(h->d_palette.p, ngp_host::ntsc_palette, sizeof(ngp_host::ntsc_palette), cudaMemcpyHostToDevice));
    NGP_CUDA(h->d_start.ensure(2));
    NGP_CUDA(h->d_counters.ensure(8));
    NGP_CUDA(cudaMemset(h->d_counters.p, 0, 8 * sizeof(unsigned long long)));
    NGP_CUDA(h->h_counters.ensure(8));
    // The two start snapshots depend on the cartridge image only: built once per process by the CUDA core (a single warp,
    // tens of milliseconds) and kept as an immutable host copy for later handles.
    {
        std::lock_guard<std::mutex> lock(g_start_mutex);
        const uint64_t key = h->cart_hash;
        auto it = g_start_cache.find(key);
        if (it == g_start_cache.end()) {
            build_start_states_kernel<<<2, 32>>>(h->d_tables.p, h->d_needed.p, h->d_start.p);
            h->launches++;
            NGP_CUDA(cudaGetLastError());
            std::vector<Snapshot> snap(2);
            NGP_CUDA(cudaMemcpy(snap.data(), h->d_start.p, 2 * sizeof(Snapshot), cudaMemcpyDeviceToHost));
            g_start_cache.emplace(key, std::move(snap));
        } else {
            NGP_CUDA(cudaMemcpy(h->d_start.p, it->second.data(), 2 * sizeof(Snapshot), cudaMemcpyHostToDevice));
        }
    }
    NGP_CUDA(cudaDeviceSynchronize());
    *out = h.release();
    return NGP_OK;
}

extern "C" int ngp_destroy(ngp_handle *h)
{
    if (!h) return NGP_OK;
    cudaSetDevice(h->device);
    delete h;
    return NGP_OK;
}

extern "C" int ngp_env_reset(ngp_handle *h, int32_t n_envs, int32_t state_id, void *stream)
{
    NGP_REQUIRE(h && n_envs > 0, "ngp_env_reset: bad arguments");
    NGP_REQUIRE(state_id == NGP_STATE_START_1P || state_id == NGP_STATE_START_2P, "ngp_env_reset: unknown state");
    NGP_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    NGP_CUDA(h->d_envs.ensure(n_envs));
    NGP_CUDA(h->d_fb.ensure((size_t)n_envs * a26::FB_ROWS * a26::FB_COLS));
    h->n_envs = n_envs;
    h->env_players = state_id == NGP_STATE_START_1P ? 1 : 2;     // main.py:40 makes the robot game with players=1
    env_reset_kernel<<<(n_envs + 127) / 128, 128, 0, st>>>(h->d_start.p + state_id, h->d_envs.p, n_envs);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}

extern "C" int ngp_env_get_state(ngp_handle *h, ngp_game_state *out, void *stream)
{
    NGP_REQUIRE(h && out, "ngp_env_get_state: bad arguments");
    NGP_REQUIRE(h->n_envs > 0, "ngp_env_get_state: call ngp_env_reset or ngp_env_set_state first");
    NGP_REQUIRE(((uintptr_t)out & 15) == 0, "ngp_env_get_state: the state array must be 16-byte aligned");
    NGP_CUDA(cudaSetDevice(h->device));
    env_get_state_kernel<<<(h->n_envs + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->d_envs.p, h->n_envs, h->env_players, h->cart_hash, out);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}

extern "C" int ngp_env_set_state(ngp_handle *h, const ngp_game_state *states, int32_t n_envs, void *stream)
{
    NGP_REQUIRE(h && states && n_envs > 0, "ngp_env_set_state: bad arguments");
    NGP_REQUIRE(((uintptr_t)states & 15) == 0, "ngp_env_set_state: the state array must be 16-byte aligned");
    NGP_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    // validate before anything is resized or written: a refused call leaves the environments as they were
    NGP_CUDA(cudaMemsetAsync(h->d_counters.p + 3, 0, 2 * sizeof(unsigned long long), st));
    state_check_kernel<<<(n_envs + 127) / 128, 128, 0, st>>>(states, n_envs, h->cart_hash, h->d_counters.p + 3);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    NGP_CUDA(cudaMemcpyAsync(h->h_counters.p + 3, h->d_counters.p + 3, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    NGP_CUDA(cudaStreamSynchronize(st));
    if (h->h_counters.p[3]) {
        ngp_set_error("ngp_env_set_state: %llu states fail validation or have another players value than the first", h->h_counters.p[3]);
        return NGP_ERR_INVALID;
    }
    NGP_CUDA(h->d_envs.ensure(n_envs));
    NGP_CUDA(h->d_fb.ensure((size_t)n_envs * a26::FB_ROWS * a26::FB_COLS));
    h->n_envs = n_envs;
    h->env_players = (int)h->h_counters.p[4];
    env_set_state_kernel<<<(n_envs + 127) / 128, 128, 0, st>>>(states, h->d_envs.p, n_envs);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}

extern "C" int ngp_env_step(ngp_handle *h, const uint8_t *actions, uint8_t *ram, uint8_t *frames, float *loc, uint8_t *valid,
                            uint8_t *regs, void *stream)
{
    return ngp_env_step_core(h, NGP_CORE_INTERPRETER, actions, ram, frames, loc, valid, regs, stream);
}

extern "C" int ngp_env_step_core(ngp_handle *h, int32_t core, const uint8_t *actions, uint8_t *ram, uint8_t *frames, float *loc,
                                 uint8_t *valid, uint8_t *regs, void *stream)
{
    NGP_REQUIRE(h && actions, "ngp_env_step: bad arguments");
    NGP_REQUIRE(h->n_envs > 0, "ngp_env_step: call ngp_env_reset first");
    NGP_REQUIRE((loc == nullptr) == (valid == nullptr), "ngp_env_step: loc and valid go together");
    if (core && !h->rom_translated) {
        ngp_set_error("ngp_env_step: the statically translated core was generated from a different cartridge; use NGP_CORE_INTERPRETER");
        return NGP_ERR_UNSUPPORTED;
    }
    NGP_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int n = h->n_envs;
    const size_t px = (size_t)n * a26::FB_ROWS * a26::FB_COLS;
    ButtonMap bmap;
    memcpy(bmap.m, h->cfg.button_map, 16);
    if (frames) NGP_CUDA(cudaMemsetAsync(h->d_fb.p, 0, px, st));
    // with a frame requested every pixel is rendered (verify mode); without, the fused no-framebuffer flavour runs
    int lanes = (n + 4 * h->sm_count - 1) / (4 * h->sm_count);           // one warp per scheduler before the warps are filled
    lanes = lanes < 1 ? 1 : (lanes > 32 ? 32 : lanes);
    const unsigned grid = (unsigned)((n + lanes - 1) / lanes);
    if (frames)
        env_step_kernel<true><<<grid, 32, 0, st>>>(h->d_tables.p, h->d_needed.p, h->d_envs.p, n, lanes, core ? 1 : 0, h->env_players, bmap, actions, h->d_fb.p,
                                                   ram, loc, valid, regs, h->d_counters.p);
    else
        env_step_kernel<false><<<grid, 32, 0, st>>>(h->d_tables.p, h->d_needed.p, h->d_envs.p, n, lanes, core ? 1 : 0, h->env_players, bmap, actions, nullptr,
                                                    ram, loc, valid, regs, h->d_counters.p);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    if (frames) {
        palette_to_rgb_kernel<<<(unsigned)((px + 255) / 256), 256, 0, st>>>(h->d_fb.p, h->d_palette.p, frames, px);
        h->launches++;
        NGP_CUDA(cudaGetLastError());
    }
    return NGP_OK;
}

extern "C" int ngp_env_digest(ngp_handle *h, uint32_t *digest, void *stream)
{
    NGP_REQUIRE(h && digest && h->n_envs > 0, "ngp_env_digest: bad arguments");
    NGP_CUDA(cudaSetDevice(h->device));
    env_digest_kernel<<<(h->n_envs + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->d_envs.p, h->n_envs, digest);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return NGP_OK;
}

// The RolloutParams fields both fused entry points fill the same way; everything else starts zero (no match list).
static RolloutParams rollout_params(const ngp_handle *h, const float *genomes, uint64_t seed, uint64_t generation)
{
    RolloutParams p = {};
    p.tables = h->d_tables.p; p.needed = h->d_needed.p; p.start = h->d_start.p;
    p.genomes = genomes; p.G = h->gene_size; p.schedule = h->cfg.schedule;
    p.core = h->cfg.core ? 1 : 0;
    p.win_score = h->cfg.win_score; p.timeout_thresh = h->cfg.timeout_thresh; p.max_frames = h->cfg.max_frames;
    p.time_scaler = (double)h->cfg.time_scaler; p.paddle_height = (double)h->cfg.scaled_paddle_height;
    p.seed = seed; p.generation = generation; p.shape = h->shape;
    roll::fill_input_table(p, h->cfg.button_map);
    p.counters = h->d_counters.p;
    return p;
}

// Launches rollout_kernel over `total` environments, between the profiling events when profiling is on.  With `rec`
// (ngp_record_matches) the recording twin of the flavour these rules pick is launched instead.
static int launch_rollout(ngp_handle *h, const RolloutParams &p, long long total, cudaStream_t st, const char *who,
                          const roll::RecordArgs *rec = nullptr)
{
    // Launch geometry (measured, profiles/README.md).  Small launches: one-warp CTAs spread over all SMs.  From ~2 warps per
    // SM upwards the CTA-synchronous flavour wins: all warps of a CTA walk through the frame together and share their
    // instruction fetches; the CTA grows with the launch until one 16-warp CTA per SM (128 registers/thread) is reached.
    int block = 32;
    long long warps = (total + 31) / 32;
    if (p.core && total >= 12288) {
        // measured at 12288 / 24576 / 49152 environments (profiles/README.md): while one CTA per SM is enough, 128- or
        // 256- / 384-thread CTAs with the largest register budget that fits; beyond that 512-thread CTAs
        if (total <= (long long)h->sm_count * 128) block = 128;
        else if (total <= (long long)h->sm_count * 256) block = 256;
        else if (total <= (long long)h->sm_count * 384) block = 384;
        else block = 512;
    } else if (!p.core && warps > (long long)h->sm_count * 16) block = 128;
    // tuning overrides (ngp_set_option; experiments and the geometry-independence tests only)
    if (h->opt_rollout_block >= 32 && h->opt_rollout_block <= 1024 && h->opt_rollout_block % 32 == 0) block = h->opt_rollout_block;
    const bool sync = p.core && block > 32 && !h->opt_rollout_nosync;
    // register budget: MAXT=256 lets the compiler have the ~210-230 registers it wants (no spills: +8 % per one-warp CTA, +22 %
    // for CTA-synchronous launches, measured); MAXT=384 gives 168, MAXT=512 caps them at 128 (16 warps per SM).
    // While every CTA has an SM to itself the fattest flavour that fits the CTA is used; beyond that occupancy is worth more
    // than the spills.
    long long blocks = (total + block - 1) / block;
    const bool one_per_sm = blocks <= (long long)h->sm_count;
    int lean = sync ? (one_per_sm && block <= 256 ? 0 : one_per_sm && block <= 384 ? 2 : 1) : 0;
    if (h->opt_rollout_lean) lean = h->opt_rollout_lean - 1;       // option value 1..3 = flavour 0 (256), 1 (512), 2 (384)
    if (!sync) lean = 0;
    if (sync && block > (lean == 0 ? 256 : lean == 2 ? 384 : 512)) lean = block > 384 ? 1 : 2;   // the flavour's launch bound must hold the CTA
    if (block > (sync ? 512 : p.core ? 256 : 384)) {
        ngp_set_error("%s: rollout_block exceeds the kernel flavour's launch bound", who);
        return NGP_ERR_INVALID;
    }
    const int flavour = !p.core ? 0 : !sync ? 1 : lean == 2 ? 3 : lean == 1 ? 4 : 2;      // rollout_record_kernel's numbering
    static const RolloutKernel flavours[5] = {rollout_kernel<0, false, 384>, rollout_kernel<1, false, 256>, rollout_kernel<1, true, 256>,
                                              rollout_kernel<1, true, 384>, rollout_kernel<1, true, 512>};
    const RolloutKernel kernel = rec ? rollout_record_kernel(flavour) : flavours[flavour];
    const size_t smem = (size_t)block * 32 * 4;
    int per_sm = 0;
    if (smem + sizeof(Tables) > 48 * 1024) NGP_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    NGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, smem));
    if (per_sm < 1) per_sm = 1;
    if (h->opt_rollout_blocks_per_sm >= 1 && h->opt_rollout_blocks_per_sm < per_sm) per_sm = h->opt_rollout_blocks_per_sm;
    const long long resident = (long long)per_sm * h->sm_count;
    if (blocks > resident) blocks = resident;            // persistent lanes pull the rest from the queue
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    if (h->profile_on) {
        if (h->prof_used == (int)h->prof_events.size()) {
            cudaEvent_t a, b;
            NGP_CUDA(cudaEventCreate(&a)); NGP_CUDA(cudaEventCreate(&b));
            h->prof_events.push_back({a, b});
        }
        ev0 = h->prof_events[h->prof_used].first; ev1 = h->prof_events[h->prof_used].second;
        h->prof_used++;
        NGP_CUDA(cudaEventRecord(ev0, st));
    }
    kernel<<<(unsigned)blocks, block, smem, st>>>(p, rec ? *rec : roll::RecordArgs{});
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    if (ev1) NGP_CUDA(cudaEventRecord(ev1, st));
    return NGP_OK;
}

// Copies the frame and error counters back (synchronises the stream); the emulator-error report of both fused entry points.
static int read_rollout_counters(ngp_handle *h, cudaStream_t st, uint64_t *frames_total, const char *who)
{
    NGP_CUDA(cudaMemcpyAsync(h->h_counters.p, h->d_counters.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    NGP_CUDA(cudaStreamSynchronize(st));
    *frames_total = h->h_counters.p[1];
    if (h->h_counters.p[2]) {
        ngp_set_error("%s: %llu environments stopped on an emulator error", who, h->h_counters.p[2]);
        return NGP_ERR_EMULATOR;
    }
    return NGP_OK;
}

extern "C" int ngp_evaluate(ngp_handle *h, const float *genomes, int32_t n, const float *hof_genomes, const double *hof_fitness,
                            int32_t n_hof, const int32_t *hof_pick, uint64_t seed, uint64_t generation, double *fitness,
                            double *rewards, int32_t *frames, uint64_t *frames_total, void *stream)
{
    NGP_REQUIRE(h && genomes && fitness && n > 0, "ngp_evaluate: bad arguments");
    NGP_REQUIRE(n_hof == 0 || (hof_genomes && hof_fitness), "ngp_evaluate: hall of fame pointers missing");
    bool wide = false;            // a layer too wide for the fused thread-per-environment MLP: per-frame stepwise driver (ngp_stepwise.cu)
    for (int i = 0; i < h->cfg.n_layers; ++i) wide |= h->cfg.nodes[i] > pol::FUSED_MAX_WIDTH;
    NGP_REQUIRE(!wide || (h->cfg.nodes[0] == 6 && h->cfg.nodes[h->cfg.n_layers - 1] <= 8),
                "ngp_evaluate: wide networks need 6 inputs and at most 8 outputs");
    if (h->cfg.schedule == NGP_SCHEDULE_REFERENCE)
        NGP_REQUIRE(h->cfg.games_to_play <= NGP_GAMES_TO_PLAY, "ngp_evaluate: the reference schedule has at most 6 games");
    NGP_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int games = h->cfg.games_to_play;
    const long long total = (long long)n * games;
    NGP_REQUIRE(total < (1ll << 31), "ngp_evaluate: too many environments");
    NGP_CUDA(h->d_rewards.ensure(total));
    NGP_CUDA(h->d_frames.ensure(total));
    NGP_CUDA(cudaMemsetAsync(h->d_counters.p, 0, 8 * sizeof(unsigned long long), st));
    RolloutParams p = rollout_params(h, genomes, seed, generation);
    p.hof_genomes = hof_genomes; p.hof_fitness = hof_fitness; p.hof_pick = hof_pick;
    p.n = n; p.n_hof = n_hof; p.games = games;
    if (p.core && !h->rom_translated) {
        ngp_set_error("ngp_evaluate: the statically translated core was generated from a different cartridge; use NGP_CORE_INTERPRETER");
        return NGP_ERR_UNSUPPORTED;
    }
    p.rewards = rewards ? rewards : h->d_rewards.p; p.frames = frames ? frames : h->d_frames.p;
    if (wide) {
        const int rc = ngp_evaluate_stepwise(h, p, st);
        if (rc != NGP_OK) return rc;
        fitness_reduce_kernel<<<(n + 127) / 128, 128, 0, st>>>(p.rewards, n, games, fitness);
        h->launches++;
        NGP_CUDA(cudaGetLastError());
        if (frames_total) *frames_total = h->h_counters.p[1];
        if (h->h_counters.p[2]) {
            ngp_set_error("ngp_evaluate: %llu environments stopped on an emulator error", h->h_counters.p[2]);
            return NGP_ERR_EMULATOR;
        }
        return NGP_OK;
    }
    const int rc = launch_rollout(h, p, total, st, "ngp_evaluate");
    if (rc != NGP_OK) return rc;
    fitness_reduce_kernel<<<(n + 127) / 128, 128, 0, st>>>(p.rewards, n, games, fitness);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    return frames_total ? read_rollout_counters(h, st, frames_total, "ngp_evaluate") : NGP_OK;
}

// ngp_play_matches; ngp_record_matches and ngp_play_matches_states when `rec` is set (its pointers' alignment and the record
// length already checked; n_states = the length of rec->states)
static int play_match_list(ngp_handle *h, const float *genomes, int32_t n_genomes, const int32_t *right, const int32_t *left,
                           const double *mult, int32_t n_matches, uint64_t seed, uint64_t generation, double *rewards, int32_t *frames,
                           int32_t *scores, uint64_t *frames_total, cudaStream_t st, const roll::RecordArgs *rec, int32_t n_states,
                           const char *who)
{
    if (!(h && genomes && right && left && rewards && n_genomes > 0 && n_matches > 0)) {
        ngp_set_error("%s: bad arguments", who);
        return NGP_ERR_INVALID;
    }
    for (int i = 0; i < h->cfg.n_layers; ++i)
        if (h->cfg.nodes[i] > pol::FUSED_MAX_WIDTH) {
            // the stepwise driver batches the MLP by genome with a fixed number of rows per genome; a match list has none
            ngp_set_error("%s: networks with a layer wider than %d units are not supported (the fused rollout only)", who,
                          pol::FUSED_MAX_WIDTH);
            return NGP_ERR_UNSUPPORTED;
        }
    if (h->cfg.core && !h->rom_translated) {
        ngp_set_error("%s: the statically translated core was generated from a different cartridge; use NGP_CORE_INTERPRETER", who);
        return NGP_ERR_UNSUPPORTED;
    }
    const roll::RecordArgs none = {};
    const roll::RecordArgs &ra = rec ? *rec : none;
    NGP_CUDA(cudaSetDevice(h->device));
    if (!frames) NGP_CUDA(h->d_frames.ensure(n_matches));
    NGP_CUDA(cudaMemsetAsync(h->d_counters.p, 0, 8 * sizeof(unsigned long long), st));
    // the lists and states live on the device: count their bad entries there and refuse before anything is played
    const long long check_items = std::max<long long>(n_matches, n_states);
    const int check_blocks = (int)std::min<long long>((check_items + 255) / 256, 4ll * h->sm_count);
    match_check_kernel<<<check_blocks, 256, 0, st>>>(right, left, ra.key, n_matches, n_genomes, ra.capture_at, ra.start, ra.states, n_states,
                                                     h->cart_hash, h->d_counters.p + 3);
    h->launches++;
    NGP_CUDA(cudaGetLastError());
    NGP_CUDA(cudaMemcpyAsync(h->h_counters.p + 3, h->d_counters.p + 3, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    NGP_CUDA(cudaStreamSynchronize(st));
    if (h->h_counters.p[3]) {
        if (ra.start || ra.capture_at || n_states)
            ngp_set_error("%s: %llu faults in the match entries (genome rows, NGP_OPP_* codes, keys, start indices, capture frames, "
                          "players of the start states) or start states that fail validation", who, h->h_counters.p[3]);
        else
            ngp_set_error(ra.key ? "%s: %llu match entries name no genome row (right), no genome row or NGP_OPP_* code (left) or a negative key"
                                 : "%s: %llu match entries name no genome row (right) or no genome row or NGP_OPP_* code (left)",
                          who, h->h_counters.p[3]);
        return NGP_ERR_INVALID;
    }
    RolloutParams p = rollout_params(h, genomes, seed, generation);
    p.n = n_matches; p.games = 1;
    p.match_right = right; p.match_left = left; p.match_mult = mult;
    p.rewards = rewards; p.frames = frames ? frames : h->d_frames.p; p.scores = scores;
    const int rc = launch_rollout(h, p, n_matches, st, who, rec);
    if (rc != NGP_OK) return rc;
    return frames_total ? read_rollout_counters(h, st, frames_total, who) : NGP_OK;
}

extern "C" int ngp_play_matches(ngp_handle *h, const float *genomes, int32_t n_genomes, const int32_t *right, const int32_t *left,
                                const double *mult, int32_t n_matches, uint64_t seed, uint64_t generation, double *rewards,
                                int32_t *frames, int32_t *scores, uint64_t *frames_total, void *stream)
{
    return play_match_list(h, genomes, n_genomes, right, left, mult, n_matches, seed, generation, rewards, frames, scores,
                           frames_total, (cudaStream_t)stream, nullptr, 0, "ngp_play_matches");
}

extern "C" int ngp_record_matches(ngp_handle *h, const float *genomes, int32_t n_genomes, const int32_t *right, const int32_t *left,
                                  const double *mult, const int32_t *key, int32_t n_matches, uint64_t seed, uint64_t generation,
                                  int32_t max_record, ngp_frame_record *record, double *rewards, int32_t *frames, int32_t *scores,
                                  uint64_t *frames_total, void *stream)
{
    NGP_REQUIRE(max_record >= 1 && record, "ngp_record_matches: needs a record buffer and max_record >= 1");
    NGP_REQUIRE(((uintptr_t)record & 15) == 0, "ngp_record_matches: the record buffer must be 16-byte aligned");
    roll::RecordArgs rec = {};
    rec.record = record; rec.key = key; rec.max_record = max_record;
    return play_match_list(h, genomes, n_genomes, right, left, mult, n_matches, seed, generation, rewards, frames, scores,
                           frames_total, (cudaStream_t)stream, &rec, 0, "ngp_record_matches");
}

extern "C" int ngp_play_matches_states(ngp_handle *h, const float *genomes, int32_t n_genomes, const int32_t *right, const int32_t *left,
                                       const double *mult, const int32_t *key, int32_t n_matches, const ngp_game_state *states,
                                       int32_t n_states, const int32_t *start, int32_t fresh, const int32_t *capture_at,
                                       ngp_game_state *capture, int32_t max_record, ngp_frame_record *record, uint64_t seed,
                                       uint64_t generation, double *rewards, int32_t *frames, int32_t *scores, uint64_t *frames_total,
                                       void *stream)
{
    NGP_REQUIRE(h, "ngp_play_matches_states: null handle");
    NGP_REQUIRE(!record || max_record >= 1, "ngp_play_matches_states: a record needs max_record >= 1");
    NGP_REQUIRE(((uintptr_t)record & 15) == 0, "ngp_play_matches_states: the record buffer must be 16-byte aligned");
    NGP_REQUIRE(n_states >= 0 && (n_states == 0 || states), "ngp_play_matches_states: n_states states needed");
    NGP_REQUIRE(((uintptr_t)states & 15) == 0 && ((uintptr_t)capture & 15) == 0, "ngp_play_matches_states: state arrays must be 16-byte aligned");
    NGP_REQUIRE(!capture_at || capture, "ngp_play_matches_states: capture_at needs a capture buffer");
    roll::RecordArgs rec = {};
    rec.record = record; rec.key = key; rec.max_record = record ? max_record : 0;
    rec.fresh = fresh ? 1 : 0; rec.states = states; rec.start = start; rec.capture_at = capture_at; rec.capture = capture;
    rec.cart = h->cart_hash;
    return play_match_list(h, genomes, n_genomes, right, left, mult, n_matches, seed, generation, rewards, frames, scores,
                           frames_total, (cudaStream_t)stream, &rec, n_states, "ngp_play_matches_states");
}

extern "C" int ngp_profile_enable(ngp_handle *h, int32_t on)
{
    NGP_REQUIRE(h, "ngp_profile_enable: null handle");
    h->profile_on = on ? 1 : 0;
    return NGP_OK;
}

extern "C" int ngp_profile_read(ngp_handle *h, double *rollout_ms, int32_t *rollout_launches)
{
    NGP_REQUIRE(h && rollout_ms && rollout_launches, "ngp_profile_read: bad arguments");
    NGP_CUDA(cudaSetDevice(h->device));
    double total = 0.0;
    for (int i = 0; i < h->prof_used; ++i) {
        float ms = 0.f;
        NGP_CUDA(cudaEventSynchronize(h->prof_events[i].second));
        NGP_CUDA(cudaEventElapsedTime(&ms, h->prof_events[i].first, h->prof_events[i].second));
        total += ms;
    }
    *rollout_ms = total;
    *rollout_launches = h->prof_used;
    h->prof_used = 0;
    return NGP_OK;
}

extern "C" int ngp_evaluate_host(ngp_handle *h, const float *genomes, int32_t n, const float *hof_genomes, const double *hof_fitness,
                                 int32_t n_hof, uint64_t seed, uint64_t generation, double *fitness, uint64_t *frames_total)
{
    NGP_REQUIRE(h && genomes && fitness && n > 0, "ngp_evaluate_host: bad arguments");
    NGP_CUDA(cudaSetDevice(h->device));
    const size_t genes = (size_t)n * h->gene_size, gbytes = genes * sizeof(float), fbytes = (size_t)n * sizeof(double);
    NGP_CUDA(h->h_genomes.ensure(genes));
    NGP_CUDA(h->d_genomes_stage.ensure(genes));
    NGP_CUDA(h->h_fitness.ensure(n));
    NGP_CUDA(h->d_fitness_stage.ensure(n));
    memcpy(h->h_genomes.p, genomes, gbytes);
    NGP_CUDA(cudaMemcpyAsync(h->d_genomes_stage.p, h->h_genomes.p, gbytes, cudaMemcpyHostToDevice, 0));
    if (n_hof > 0) {
        const size_t hof_genes = (size_t)n_hof * h->gene_size;
        NGP_CUDA(h->d_hof_stage.ensure(hof_genes));
        NGP_CUDA(h->d_hof_fit_stage.ensure(n_hof));
        NGP_CUDA(cudaMemcpyAsync(h->d_hof_stage.p, hof_genomes, hof_genes * sizeof(float), cudaMemcpyHostToDevice, 0));
        NGP_CUDA(cudaMemcpyAsync(h->d_hof_fit_stage.p, hof_fitness, (size_t)n_hof * sizeof(double), cudaMemcpyHostToDevice, 0));
    }
    uint64_t ft = 0;
    int rc = ngp_evaluate(h, h->d_genomes_stage.p, n, n_hof ? h->d_hof_stage.p : nullptr, n_hof ? h->d_hof_fit_stage.p : nullptr, n_hof,
                          nullptr, seed, generation, h->d_fitness_stage.p, nullptr, nullptr, &ft, 0);
    if (rc != NGP_OK) return rc;
    NGP_CUDA(cudaMemcpyAsync(h->h_fitness.p, h->d_fitness_stage.p, fbytes, cudaMemcpyDeviceToHost, 0));
    NGP_CUDA(cudaStreamSynchronize(0));
    memcpy(fitness, h->h_fitness.p, fbytes);
    if (frames_total) *frames_total = ft;
    return NGP_OK;
}
