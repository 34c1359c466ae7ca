// Sanitizer fuzz driver for the multichannel Vorbis front-end (symgpu_vorbis_fe_*_mc):
//   g++ -std=c++17 -O1 -g -fsanitize=address,undefined -fno-sanitize-recover=all ... tests/cpp/fuzz_vorbis_mc.cpp vorbis_frontend.cpp packetizer.cpp tables.cpp
//   fuzz_vorbis_mc SEEDFILE... : a seed is [u16 length, bytes]... = identification header, setup header, audio packets.  Every seed is
// mutated (bit flips, byte runs, truncation, splices) ITER times and pushed through create_mc / config_mc / decode_mc (at the stream's
// channel count and at 8 planes), decode_packets_mc and decode_packets_jobs_mc; any out-of-bounds access, overflow or leak aborts.
// Run by tests/test_vorbis_multichannel.py.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <random>
#include <vector>

#include "../../include/symgpu.h"

static void run_all(const std::vector<uint8_t>& d) {
    const uint8_t* p = d.data();
    const size_t n = d.size();
    std::vector<symgpu_piece> parts;
    size_t at = 0;
    while (at + 2 <= n) {
        const size_t len = size_t(p[at]) | size_t(p[at + 1]) << 8;
        at += 2;
        const size_t take = len < n - at ? len : n - at;
        parts.push_back(symgpu_piece{at, uint32_t(take), 0});
        at += take;
    }
    if (parts.size() < 2) return;
    const uint8_t *ident = p + parts[0].offset, *setup = p + parts[1].offset;
    const std::vector<symgpu_piece> tab(parts.begin() + 2, parts.end());
    symgpu_vorbis_fe* fe = nullptr;
    if (symgpu_vorbis_fe_create_mc(ident, parts[0].len, setup, parts[1].len, &fe) != SYMGPU_OK) return;
    symgpu_vorbis_stream_mc st;
    std::vector<symgpu_vorbis_floor1> fl(64);
    uint32_t nf = 0;
    symgpu_vorbis_fe_config_mc(fe, &st, fl.data(), &nf);
    const uint32_t slot = (1u << st.bs1_exp) >> 1;
    for (uint32_t planes : {uint32_t(st.channels), uint32_t(SYMGPU_VORBIS_MAX_CHANNELS)}) {
        std::vector<uint16_t> fy(65 * size_t(planes) * (tab.size() + 1));
        std::vector<float> res(size_t(planes) * slot * (tab.size() + 1));
        std::vector<symgpu_vorbis_unit_mc> u(tab.size() + 1);
        for (size_t k = 0; k < tab.size(); ++k) {
            symgpu_vorbis_fe_decode_mc(fe, p + tab[k].offset, tab[k].len, slot, 0, planes, u.data(), fy.data(), res.data());
            if (k % 5 == 0) symgpu_vorbis_fe_reset(fe);
        }
        std::vector<uint32_t> idx(tab.size() + 1);
        size_t good = 0;
        symgpu_vorbis_fe_decode_packets_mc(fe, p, n, tab.data(), tab.size(), slot, 0, planes, u.data(), fy.data(), res.data(), idx.data(), &good);
        if (tab.size() < 200)
            symgpu_vorbis_fe_decode_packets_jobs_mc(ident, parts[0].len, setup, parts[1].len, p, n, tab.data(), tab.size(), slot, 0, planes, u.data(),
                                                    fy.data(), res.data(), idx.data(), &good, 2);
    }
    symgpu_vorbis_fe_destroy(fe);
}

int main(int argc, char** argv) {
    const int iters = std::getenv("FUZZ_ITERS") ? std::atoi(std::getenv("FUZZ_ITERS")) : 200;
    std::mt19937_64 rng(4321);
    size_t runs = 0;
    for (int a = 1; a < argc; ++a) {
        std::ifstream in(argv[a], std::ios::binary);
        const std::vector<uint8_t> seed((std::istreambuf_iterator<char>(in)), std::istreambuf_iterator<char>());
        run_all(seed), ++runs;
        for (int it = 0; it < iters && !seed.empty(); ++it) {
            std::vector<uint8_t> d = seed;
            const int kinds = 1 + int(rng() % 3);
            for (int k = 0; k < kinds; ++k) {
                const size_t at = rng() % d.size();
                switch (rng() % 5) {
                    case 0: d[at] ^= uint8_t(1u << (rng() % 8)); break;
                    case 1: d[at] = uint8_t(rng()); break;
                    case 2: {
                        const size_t len = std::min<size_t>(1 + rng() % 16, d.size() - at);
                        std::memset(d.data() + at, (rng() & 1) ? 0xff : 0x00, len);
                        break;
                    }
                    case 3: d.resize(1 + at); break;
                    default: {
                        const size_t from = rng() % d.size(), len = std::min<size_t>(1 + rng() % 64, std::min(d.size() - from, d.size() - at));
                        std::memmove(d.data() + at, d.data() + from, len);
                    }
                }
                if (d.empty()) break;
            }
            if (!d.empty()) run_all(d), ++runs;
        }
    }
    std::printf("fuzz: %zu inputs, no sanitizer report\n", runs);
    return 0;
}
