// host_tables.h -- host-side construction of the constant tables the kernels read
#pragma once
#include <stdint.h>
#include <string.h>

#include "../../include/ngp.h"
#include "a26_compiled.cuh"

namespace ngp_host {

// Stella NTSC palette [3P-recall]; entries $0E,$22,$38,$C8 are pinned by config.py:3-6 + obs.npy
inline constexpr uint32_t ntsc_palette[128] = {
    0x000000, 0x4a4a4a, 0x6f6f6f, 0x8e8e8e, 0xaaaaaa, 0xc0c0c0, 0xd6d6d6, 0xececec, 0x484800, 0x69690f, 0x86861d, 0xa2a22a,
    0xbbbb35, 0xd2d240, 0xe8e84a, 0xfcfc54, 0x7c2c00, 0x904811, 0xa26221, 0xb47a30, 0xc3903d, 0xd2a44a, 0xdfb755, 0xecc860,
    0x901c00, 0xa33915, 0xb55328, 0xc66c3a, 0xd5824a, 0xe39759, 0xf0aa67, 0xfcbc74, 0x940000, 0xa71a1a, 0xb83232, 0xc84848,
    0xd65c5c, 0xe46f6f, 0xf08080, 0xfc9090, 0x840064, 0x97197a, 0xa8308f, 0xb846a2, 0xc659b3, 0xd46cc3, 0xe07cd2, 0xec8ce0,
    0x500084, 0x68199a, 0x7d30ad, 0x9246c0, 0xa459d0, 0xb56ce0, 0xc57cee, 0xd48cfc, 0x140090, 0x331aa3, 0x4e32b5, 0x6848c6,
    0x7f5cd5, 0x956fe3, 0xa980f0, 0xbc90fc, 0x000094, 0x181aa7, 0x2d32b8, 0x4248c8, 0x545cd6, 0x656fe4, 0x7580f0, 0x8490fc,
    0x001c88, 0x183b9d, 0x2d57b0, 0x4272c2, 0x548ad2, 0x65a0e1, 0x75b5ef, 0x84c8fc, 0x003064, 0x185080, 0x2d6d98, 0x4288b0,
    0x54a0c5, 0x65b7d9, 0x75cceb, 0x84e0fc, 0x004030, 0x18624e, 0x2d8169, 0x429e82, 0x54b899, 0x65d1ae, 0x75e7c2, 0x84fcd4,
    0x004400, 0x1a661a, 0x328432, 0x48a048, 0x5cba5c, 0x6fd26f, 0x80e880, 0x90fc90, 0x143c00, 0x355f18, 0x527e2d, 0x6e9c42,
    0x87b754, 0x9ed065, 0xb4e775, 0xc8fc84, 0x303800, 0x505916, 0x6d762b, 0x88923e, 0xa0ab4f, 0xb7c25f, 0xccd86e, 0xe0ec7c,
    0x482c00, 0x694d14, 0x866a26, 0xa28638, 0xbb9f47, 0xd2b656, 0xe8cc63, 0xfce070,
};

// ngp_default_config's button map: the reference's own naming (config.py:15-20, main.py:91-92) -- see include/ngp.h
inline void default_button_map(uint8_t m[16])
{
    memset(m, 0, 16);
    m[0] = NGP_BTN_FIRE_P0 + 1;      // RIGHT_PLAYER_START_BUTTON = 0
    m[15] = NGP_BTN_FIRE_P0 + 0;     // LEFT_PLAYER_START_BUTTON = -1
    m[4] = NGP_BTN_UP_P0 + 2; m[5] = NGP_BTN_UP_P0 + 3;      // action[4:6]: right player = paddle 1
    m[6] = NGP_BTN_UP_P0 + 0; m[7] = NGP_BTN_UP_P0 + 1;      // action[6:8]: left player = paddle 0
    m[2] = m[10] = NGP_BTN_SELECT;
    m[3] = m[11] = NGP_BTN_RESET;
}

// Stella TIA::dumpedInputPort / Paddles::update [3P-recall]: resistance = 1.4e6 * charge/4096,
// CPU cycles until INPTx bit 7 rises = 1.216e-6 * resistance * scanlines(262) * framerate(59.92)
inline void build_paddle_table(uint32_t *t)
{
    for (int c = 0; c <= a26::TRIGMAX; ++c) {
        int32_t resistance = (int32_t)(1400000 * (c / (float)a26::TRIGMAX));
        t[c] = (uint32_t)(1.216e-6 * resistance * 262.0 * 59.92f);
    }
}

// rom words + decode table + per-palette-entry colour-match weights: 2 bits per target colour =
// number of RGB channels of the palette entry equal to the target's (the reference matches per
// channel, utils.py:62)
inline void build_tables(a26::Tables &tables, const uint8_t *rom, const uint8_t ball[3], const uint8_t left[3],
                         const uint8_t right[3], const uint32_t palette[128])
{
    memset(&tables, 0, sizeof(tables));
    memcpy(tables.rom, rom, 2048);
    a26::DecodeTable dt;
    a26::build_decode_table(dt);
    memcpy(tables.decode, dt.e, sizeof(dt.e));
    a26::fill_blockmap(tables.blockmap);
    const uint8_t *targets[3] = {ball, left, right};
    for (int i = 0; i < 128; ++i) {
        uint32_t c = palette[i];
        uint8_t rgb[3] = {(uint8_t)(c >> 16), (uint8_t)(c >> 8), (uint8_t)c};
        uint8_t w = 0;
        for (int t = 0; t < 3; ++t) {
            int m = 0;
            for (int ch = 0; ch < 3; ++ch) m += rgb[ch] == targets[t][ch];
            w |= (uint8_t)(m << (2 * t));
        }
        tables.weight[i] = w;
    }
}

}  // namespace ngp_host
