// Vorbis entropy front-end (include/symgpu.h "Vorbis entropy front-end", SURVEY §8f N1): codebooks, floor-1 packet
// decode, residue decode and the packet-level bookkeeping of VorbisDecoder::decode_inner up to -- not including --
// inverse coupling (symphonia-codec-vorbis/src/{codebook,floor,residue,lib}.rs).  Output: what symgpu_vorbis_synth_*
// (two planes) or symgpu_vorbis_mc_synth_* (up to eight) reads.  CPU only.
//
// Floating point, bit-exact by construction: a VQ table value is `m * delta + min (+ last)` in f32 in that order, a
// residue element the running f32 sum of the vectors laid over it in pass order -- the same single IEEE operations in
// the same order as the reference (the Makefile compiles host code with -ffp-contract=off).  float32_unpack follows the
// reference down to its use of powi: 2^e is built by repeated squaring in f32 (what llvm.powi lowers to), so that
// exponents outside f32's range give the same 0 / inf the Rust gives, not ldexp's denormals.
#include <algorithm>
#include <cstring>
#include <memory>
#include <new>
#include <thread>
#include <vector>

#include "../../include/symgpu.h"
#include "../../include/symgpu/packetizer.hpp"

namespace {

using namespace symgpu::packet;

float powi2(int b) {  // compiler-rt __powisf2(2.0f, b)
    const bool recip = b < 0;
    float a = 2.0f, r = 1.0f;
    for (;;) {
        if (b & 1) r *= a;
        b /= 2;
        if (b == 0) break;
        a *= a;
    }
    return recip ? 1.0f / r : r;
}
float float32_unpack(uint32_t x) {  // codebook.rs:16-27
    const float value = float(x & 0x1fffff) * powi2(int((x & 0x7fe00000) >> 21) - 788);
    return (x & 0x80000000u) ? -value : value;
}

// The reference's BitReaderRtl, state for state (symphonia-core/src/io/bit.rs:941-1027, :1211-1250, :1305-1370).  In a Vorbis audio
// packet running out of bits is legal and decoding CONTINUES (the next channel's floor, the next sub-map's residue), so which
// bits a failed read leaves behind is observable: the reference keeps a 64-bit cache that it refills 8 bytes at a time, a read
// that fails on the FIRST refill consumes nothing, one that fails on a later refill has already dropped the cache it started
// with.  A simpler reader would differ on truncated packets; this one follows the cache.
struct PacketBits {
    const uint8_t* p;
    size_t n;         // bytes not yet fetched
    uint64_t bits = 0;
    uint32_t left = 0;
    PacketBits(const uint8_t* data, size_t len) : p(data), n(len) {}
    bool fetch() {  // fetch_bits: replace the cache with the next (up to) 8 bytes
        const size_t k = n < 8 ? n : 8;
        if (k == 0) return false;
        uint64_t v = 0;
        for (size_t i = 0; i < k; ++i) v |= uint64_t(p[i]) << (8 * i);
        p += k, n -= k, bits = v, left = uint32_t(8 * k);
        return true;
    }
    void top_up() {  // fetch_bits_partial: fill the free whole bytes of the cache
        size_t k = (64 - left) >> 3;
        if (k > n) k = n;
        for (size_t i = 0; i < k; ++i) bits |= uint64_t(p[i]) << left, left += 8;
        p += k, n -= k;
    }
    void consume(uint32_t w) { left -= w, bits = w < 64 ? bits >> w : 0; }
    bool read(uint32_t width, uint32_t& out) {  // read_bits_leq32
        uint64_t acc = bits;
        uint32_t needed = width;
        while (needed > left) {
            needed -= left;
            if (!fetch()) return false;
            acc |= bits << (width - needed);
        }
        consume(needed);
        out = uint32_t(acc & (width >= 32 ? 0xffffffffull : ((1ull << width) - 1)));
        return true;
    }
    bool read_bool(bool& out) {
        if (left < 1 && !fetch()) return false;
        out = bits & 1;
        consume(1);
        return true;
    }
};

struct Codebook {
    uint16_t dims = 0;
    bool has_vq = false;
    std::vector<float> vq;           // [entries][dims]
    std::vector<int32_t> child;      // binary trie: child[2 * node + bit] = node index, or ~value for a leaf, or 0 = no such code
    uint32_t max_len = 0;
    uint32_t lut[1024] = {};         // next ten stream bits (first bit = bit 0) -> (value + 1) << 6 | length, 0 = a longer code
    // One codeword, first stream bit = root of the tree (codebook.rs:366-369 "BitOrder::Reverse"; bit.rs:1211-1250): the cache is
    // topped up, the code is matched against it padded with zeros, and must then fit in what the cache really holds -- else the
    // packet has ended and nothing is consumed.
    bool read(PacketBits& bs, uint32_t& value) const {
        if (bs.left < max_len) bs.top_up();
        const uint32_t e = lut[bs.bits & 1023];  // codes of up to ten bits: one look-up (the cache holds zeros above `left`)
        if (e) {
            const uint32_t len = e & 63;
            if (len > bs.left) return false;
            bs.consume(len);
            return value = (e >> 6) - 1, true;
        }
        int32_t node = 0;
        for (uint32_t depth = 0; depth < 64; ++depth) {
            const uint32_t bit = uint32_t(bs.bits >> depth) & 1;
            const int32_t next = child[size_t(2 * node) + bit];
            if (next < 0) {
                if (depth + 1 > bs.left) return false;
                bs.consume(depth + 1);
                return value = uint32_t(~next), true;
            }
            if (next == 0) return false;  // cannot happen in a fully specified tree
            node = next;
        }
        return false;
    }
};

// Canonical codeword assignment (Vorbis I 3.2.1): each entry, in order, takes the lowest-valued free leaf of its length.
// Free sub-trees are kept as (prefix, depth); the tree must end up exactly full.  codebook.rs:112-210.
bool assign_codewords(const std::vector<uint8_t>& lens, std::vector<uint32_t>& words) {
    struct Free {
        uint32_t prefix;
        uint8_t depth;
    };
    std::vector<Free> free_nodes{{0, 0}};
    words.clear();
    for (uint8_t len : lens) {
        if (len == 0) continue;  // unused entries carry no codeword (the reference skips them and pushes nothing)
        int best = -1;
        uint64_t best_value = ~0ull;
        for (size_t k = 0; k < free_nodes.size(); ++k) {
            if (free_nodes[k].depth > len) continue;
            const uint64_t v = uint64_t(free_nodes[k].prefix) << (len - free_nodes[k].depth);  // its left-most leaf at this length
            if (v < best_value) best_value = v, best = int(k);
        }
        if (best < 0) return false;  // over-specified
        const Free f = free_nodes[size_t(best)];
        free_nodes.erase(free_nodes.begin() + best);
        for (uint8_t d = uint8_t(f.depth + 1); d <= len; ++d)  // going down left, every right sibling becomes free
            free_nodes.push_back(Free{uint32_t(((uint64_t(f.prefix) << (d - f.depth)) | 1)), d});
        words.push_back(uint32_t(best_value));
    }
    return free_nodes.empty();  // anything left: under-specified
}

// codebook.rs:214-360.  0 ok, 1 decode error.
int read_codebook(BitReaderRtl& bs, Codebook& cb) {
    if (bs.read(24) != 0x564342 || !bs.ok()) return 1;
    const uint32_t dims = bs.read(16), entries = bs.read(24);
    if (!bs.ok() || dims == 0 || dims > 32 || entries > 128 * 1024) return 1;
    cb.dims = uint16_t(dims);
    std::vector<uint8_t> lens;
    std::vector<uint32_t> values;
    if (!bs.read_bool()) {
        if (bs.read_bool()) {  // sparse
            for (uint32_t e = 0; e < entries && bs.ok(); ++e)
                if (bs.read_bool()) lens.push_back(uint8_t(bs.read(5) + 1)), values.push_back(e);
        } else {
            for (uint32_t e = 0; e < entries && bs.ok(); ++e) lens.push_back(uint8_t(bs.read(5) + 1)), values.push_back(e);
        }
    } else {
        uint32_t cur = 0, len = bs.read(5) + 1;
        for (;;) {
            const uint32_t num = bs.read(entries > cur ? vorbis_ilog(entries - cur) : 0);
            if (!bs.ok() || cur + num > entries) return 1;
            if (len > 32) return 1;  // (the reference would index past its 33-entry table)
            lens.insert(lens.end(), num, uint8_t(len));
            ++len, cur += num;
            if (cur == entries) break;
        }
        for (uint32_t e = 0; e < cur; ++e) values.push_back(e);
    }
    if (!bs.ok()) return 1;
    if (lens.size() == 1 && lens[0] == 1) lens.push_back(1), values.push_back(values[0]);  // single-entry book: both 1-bit codes (errata 20150226)
    const uint32_t lookup = bs.read(4);
    if (!bs.ok() || lookup > 2) return 1;
    if (lookup) {
        const float min_value = float32_unpack(bs.read(32)), delta = float32_unpack(bs.read(32));
        const uint32_t value_bits = bs.read(4) + 1;
        const bool sequence = bs.read_bool();
        if (!bs.ok()) return 1;
        uint32_t n_values;
        if (lookup == 1) {  // greatest v with v^dims <= entries (the reference computes it in f32 and asserts this bound)
            uint32_t v = 0;
            for (;;) {
                uint64_t pw = 1;
                bool over = false;
                for (uint32_t k = 0; k < dims && !over; ++k) pw *= uint64_t(v) + 1, over = pw > entries;
                if (over) break;
                ++v;
            }
            n_values = v;
        } else {
            n_values = entries * dims;
        }
        std::vector<uint16_t> mult(n_values);
        for (uint32_t k = 0; k < n_values; ++k) mult[k] = uint16_t(bs.read(value_bits));
        if (!bs.ok()) return 1;
        cb.has_vq = true;
        cb.vq.assign(size_t(entries) * dims, 0.0f);
        for (uint32_t e = 0; e < entries; ++e) {
            float last = 0.0f;
            uint32_t divisor = 1;
            for (uint32_t d = 0; d < dims; ++d) {
                const size_t at = lookup == 1 ? size_t((e / divisor) % n_values) : size_t(e) * dims + d;
                const float v = float(mult[at]) * delta + min_value + last;
                cb.vq[size_t(e) * dims + d] = v;
                if (sequence) last = v;
                divisor *= n_values;  // u32 wrap-around included, as in the reference
            }
        }
    }
    std::vector<uint32_t> words;
    if (!assign_codewords(lens, words)) return 1;
    cb.child.assign(2, 0);
    cb.max_len = lens.empty() ? 0 : *std::max_element(lens.begin(), lens.end());
    size_t w = 0;
    for (size_t k = 0; k < lens.size(); ++k) {
        if (lens[k] == 0) continue;
        int32_t node = 0;
        for (int b = lens[k] - 1; b >= 0; --b) {
            const uint32_t bit = (words[w] >> b) & 1;
            int32_t& slot = cb.child[size_t(2 * node) + bit];
            if (b == 0) {
                slot = ~int32_t(values[k]);
            } else {
                if (slot == 0) {
                    const int32_t fresh = int32_t(cb.child.size() / 2);
                    cb.child.push_back(0), cb.child.push_back(0);
                    cb.child[size_t(2 * node) + bit] = fresh;  // (push_back may have moved the storage: index again)
                    node = fresh;
                } else {
                    node = slot;
                }
            }
        }
        if (lens[k] <= 10) {
            uint32_t first = 0;  // the codeword in stream order: bit i of the index = the i-th bit read
            for (int i = 0; i < lens[k]; ++i) first |= ((words[w] >> (lens[k] - 1 - i)) & 1u) << i;
            for (uint32_t rest = 0; rest < (1u << (10 - lens[k])); ++rest) cb.lut[first | (rest << lens[k])] = (uint32_t(values[k]) + 1) << 6 | lens[k];
        }
        ++w;
    }
    return 0;
}

}  // namespace

struct symgpu_vorbis_fe {
    VorbisIdent ident{};
    VorbisSetup setup;
    std::vector<Codebook> books;
    bool stereo = false;                // what symgpu_vorbis_fe_create accepts: the two-plane entry points may decode it
    int prev_block_flag = -1;
    std::vector<float> type2;
    std::vector<uint8_t> part_classes;  // persistent across packets, see read_residue
};

namespace {

// floor.rs:655-722.  Returns false when the floor is unused (flag clear, or the packet ended inside it).
bool read_floor1(const symgpu_vorbis_fe& fe, const VorbisFloor1Setup& f, PacketBits& bs, uint16_t* y) {
    bool used;
    if (!bs.read_bool(used) || !used) return false;
    static const uint32_t ranges[4] = {256, 128, 86, 64};
    const uint32_t bits = vorbis_ilog(ranges[f.multiplier - 1] - 1);
    uint32_t v;
    if (!bs.read(bits, v)) return false;
    y[0] = uint16_t(v);
    if (!bs.read(bits, v)) return false;
    y[1] = uint16_t(v);
    int offset = 2;
    for (int p = 0; p < f.partitions; ++p) {
        const auto& cl = f.classes[f.partition_class[p]];
        const uint32_t cbits = cl.subclass_bits, csub = (1u << cbits) - 1;
        uint32_t cval = 0;
        if (cbits && !fe.books[cl.mainbook].read(bs, cval)) return false;
        for (int d = 0; d < cl.dimensions; ++d) {
            const uint32_t sub = cval & csub;
            cval >>= cbits;
            v = 0;
            if (cl.subbook_used & (1u << sub))
                if (!fe.books[cl.subbooks[sub]].read(bs, v)) return false;
            y[offset + d] = uint16_t(v);
        }
        offset += cl.dimensions;
    }
    return true;
}

// residue.rs:451-477
void decode_classes(uint32_t val, unsigned per_word, uint32_t classifications, uint8_t* out, size_t n_out) {
    unsigned skip = 0;
    if (per_word > n_out) {
        skip = unsigned(per_word - n_out);
        for (unsigned k = 0; k < skip; ++k) val /= classifications;
    }
    for (size_t k = per_word - skip; k-- > 0;) out[k] = uint8_t(val % classifications), val /= classifications;
}

// One partition: residue.rs:479-543.  false: the packet ended (legal: decoding stops), `bad` set: malformed setup.
bool read_partition(const Codebook& book, PacketBits& bs, float* out, size_t n, bool format0, bool& bad) {
    if (!book.has_vq) return bad = true, false;  // "vorbis: not a vq codebook"
    const size_t dim = book.dims;
    if (format0) {
        const size_t step = n / dim;
        for (size_t i = 0; i < step; ++i) {
            uint32_t e;
            if (!book.read(bs, e)) return false;
            const float* v = book.vq.data() + size_t(e) * dim;
            for (size_t k = 0, o = i; k < dim && o < n; ++k, o += step) out[o] += v[k];
        }
    } else {
        for (size_t o = 0; o + dim <= n; o += dim) {
            uint32_t e;
            if (!book.read(bs, e)) return false;
            const float* v = book.vq.data() + size_t(e) * dim;
            for (size_t k = 0; k < dim; ++k) out[o + k] += v[k];
        }
    }
    return true;
}

// residue.rs:142-449 for the channels in `chans` (1 to 8 of them).  0 ok, 1 decode error.
int read_residue(symgpu_vorbis_fe& fe, const VorbisResidueSetup& r, PacketBits& bs, unsigned bs_exp, const int* chans, int n_chans,
                 const uint8_t* do_not_decode, float* residue, uint32_t slot) {
    const Codebook& class_book = fe.books[r.classbook];
    const size_t n2 = (size_t(1) << bs_exp) >> 1;
    const size_t full = r.type == 2 ? n2 * size_t(n_chans) : n2;
    const size_t begin = std::min<size_t>(r.begin, full), end = std::min<size_t>(r.end, full);
    const size_t part_size = r.partition_size, per_word = class_book.dims, parts = (end - begin) / part_size;
    bool any = false;
    for (int c = 0; c < n_chans; ++c) any |= !do_not_decode[chans[c]];
    float* target[SYMGPU_VORBIS_MAX_CHANNELS] = {};
    if (r.type == 2) {
        fe.type2.assign(full, 0.0f);
    } else {
        for (int c = 0; c < n_chans; ++c) target[c] = residue + size_t(chans[c]) * slot;  // already zeroed by the caller
    }
    // the partition classes live in a vector that only ever grows and is never cleared (residue.rs:434-441): what a class word
    // writes is bounded by the vector's END, not by this packet's partition count, so a class word of the last group can spill
    // into the next channel's entries and stale entries of earlier packets stay behind -- reproduced, because later passes read them
    {
        const size_t class_slots = r.type == 2 ? parts : parts * size_t(n_chans);
        if (fe.part_classes.size() < class_slots) fe.part_classes.resize(class_slots, 0);
    }
    if (any) {
        bool bad = false, ended = false;
        for (unsigned pass = 0; pass <= r.max_pass && !ended; ++pass)
            for (size_t first = 0; first < parts && !ended; first += per_word) {
                if (pass == 0)
                    for (int c = 0; c < (r.type == 2 ? 1 : n_chans) && !ended; ++c) {
                        if (r.type != 2 && do_not_decode[chans[c]]) continue;
                        uint32_t code;
                        if (!class_book.read(bs, code)) {
                            ended = true;
                            break;
                        }
                        const size_t base = first + size_t(c) * parts;
                        decode_classes(code, unsigned(per_word), r.classifications, fe.part_classes.data() + base, fe.part_classes.size() - base);
                    }
                const size_t last = std::min(parts, first + per_word);
                for (size_t part = first; part < last && !ended; ++part)
                    for (int c = 0; c < (r.type == 2 ? 1 : n_chans) && !ended; ++c) {
                        if (r.type != 2 && do_not_decode[chans[c]]) continue;
                        const uint8_t cls = fe.part_classes[part + parts * size_t(c)];
                        if (!(r.used[cls] & (1u << pass))) continue;
                        const size_t start = begin + part_size * part;
                        float* out = (r.type == 2 ? fe.type2.data() : target[c]) + start;
                        if (!read_partition(fe.books[r.books[cls][pass]], bs, out, part_size, r.type == 0, bad)) ended = true;
                    }
            }
        if (bad) return 1;
    }
    if (r.type == 2)  // de-interleave (residue.rs:177-218)
        for (int c = 0; c < n_chans; ++c) {
            float* out = residue + size_t(chans[c]) * slot;
            for (size_t i = 0; i < n2; ++i) out[i] = fe.type2[i * size_t(n_chans) + size_t(c)];
        }
    return 0;
}

}  // namespace

namespace {

// Headers -> front-end, with what both create entry points refuse.  Sets fe->stereo when the stream is one the two-plane synthesis
// takes: at most two channels and every mapping uncoupled or coupled by the one step (0, 1), the same number of steps in every mode.
symgpu_status open_stream(const uint8_t* ident, size_t n_ident, const uint8_t* setup, size_t n_setup, std::unique_ptr<symgpu_vorbis_fe>& fe) {
    if (!ident || !setup) return SYMGPU_ERR_ARG;
    fe.reset(new (std::nothrow) symgpu_vorbis_fe());
    if (!fe) return SYMGPU_ERR_LIMIT;
    const Status si = vorbis_read_ident(ident, n_ident, fe->ident);
    if (si != Status::Ok) return si == Status::Unsupported ? SYMGPU_ERR_UNSUPPORTED : SYMGPU_ERR_DECODE;
    if (vorbis_read_setup(setup, n_setup, fe->ident, fe->setup) != Status::Ok) return SYMGPU_ERR_DECODE;
    // the codebooks once more, this time built (the walk above only checked their syntax)
    BitReaderRtl bs(setup + 7, n_setup - 7);
    const uint32_t n_books = bs.read(8) + 1;
    fe->books.resize(n_books);
    for (uint32_t k = 0; k < n_books; ++k)
        if (read_codebook(bs, fe->books[k])) return SYMGPU_ERR_DECODE;
    // residue partitions must fit the blocks they are laid over (the reference would panic slicing past the vector)
    // -- checked per packet; here: what the synthesis kernels cannot take.  The reference has no channel map beyond 8 (lib.rs:771-788).
    if (fe->ident.n_channels > SYMGPU_VORBIS_MAX_CHANNELS) return SYMGPU_ERR_UNSUPPORTED;
    for (uint8_t t : fe->setup.floor_type)
        if (t != 1) return SYMGPU_ERR_UNSUPPORTED;
    bool stereo = fe->ident.n_channels <= 2;
    for (const auto& m : fe->setup.mappings) {
        if (m.couplings.size() > SYMGPU_VORBIS_MAX_COUPLINGS) return SYMGPU_ERR_UNSUPPORTED;
        if (m.couplings.size() > 1) stereo = false;
        if (m.couplings.size() == 1 && !(m.couplings[0].first == 0 && m.couplings[0].second == 1)) stereo = false;
    }
    // what symgpu_vorbis_floors_set will insist on at launch time is refused here, per stream (a setup whose read X values
    // repeat an implied end point passes the reference's parser but would divide by zero in its render_line)
    {
        std::vector<symgpu_vorbis_floor1> fl(fe->setup.floor1.size());
        for (size_t i = 0; i < fl.size(); ++i) {
            const VorbisFloor1Setup& f = fe->setup.floor1[i];
            std::memset(&fl[i], 0, sizeof fl[i]);
            fl[i].multiplier = f.multiplier, fl[i].n_posts = f.n_posts;
            std::memcpy(fl[i].x_list, f.x_list, sizeof fl[i].x_list), std::memcpy(fl[i].low, f.low, 65), std::memcpy(fl[i].high, f.high, 65),
                std::memcpy(fl[i].sort_order, f.sort_order, 65);
        }
        if (!fl.empty() && symgpu_vorbis_floors_check(fl.data(), uint32_t(fl.size())) != SYMGPU_OK) return SYMGPU_ERR_UNSUPPORTED;
    }
    // one coupling record per stream: the two-plane record holds a flag (every mode's mapping must agree on the step count), the
    // multichannel record a list (every mode's mapping must have the same list)
    const auto& first = fe->setup.mappings[fe->setup.modes[0].second].couplings;
    bool same_lists = true;
    for (size_t k = 1; k < fe->setup.modes.size(); ++k) {
        const auto& c = fe->setup.mappings[fe->setup.modes[k].second].couplings;
        if (c.size() != first.size()) stereo = false;
        if (c != first) same_lists = false;
    }
    fe->stereo = stereo;  // (implies same_lists)
    return same_lists ? SYMGPU_OK : SYMGPU_ERR_UNSUPPORTED;
}

void floor_records(const symgpu_vorbis_fe* fe, symgpu_vorbis_floor1* floors, uint32_t* n_floors) {
    *n_floors = uint32_t(fe->setup.floor1.size());
    for (size_t i = 0; i < fe->setup.floor1.size(); ++i) {
        const VorbisFloor1Setup& f = fe->setup.floor1[i];
        symgpu_vorbis_floor1& o = floors[i];
        std::memset(&o, 0, sizeof o);
        o.multiplier = f.multiplier, o.n_posts = f.n_posts;
        std::memcpy(o.x_list, f.x_list, sizeof o.x_list), std::memcpy(o.low, f.low, 65), std::memcpy(o.high, f.high, 65), std::memcpy(o.sort_order, f.sort_order, 65);
    }
}

// One audio packet into `planes` channel planes (floor_y [planes][65], residue [planes][slot]); the stereo and multichannel entry points
// both come here.  Planes beyond the stream's channels are zero, marked not decoded and without a floor.
symgpu_status decode_packet(symgpu_vorbis_fe* fe, const uint8_t* packet, size_t n, uint32_t slot, uint32_t floor_base, uint32_t planes,
                            symgpu_vorbis_unit_mc* unit, uint16_t* floor_y, float* residue) {
    PacketBits bs(packet, n);
    bool flag;
    if (!bs.read_bool(flag) || flag) return SYMGPU_ERR_DECODE;  // lib.rs:151-154
    const size_t n_modes = fe->setup.modes.size();
    uint32_t mode_number;
    if (!bs.read(vorbis_ilog(uint32_t(n_modes - 1)), mode_number) || mode_number >= n_modes) return SYMGPU_ERR_DECODE;
    const bool long_block = fe->setup.modes[mode_number].first;
    const VorbisMappingSetup& mapping = fe->setup.mappings[fe->setup.modes[mode_number].second];
    if (long_block) {  // previous / next window flags: read, not used (lib.rs:168-173)
        if (!bs.read_bool(flag) || !bs.read_bool(flag)) return SYMGPU_ERR_DECODE;
    }
    const unsigned bs_exp = long_block ? fe->ident.bs1_exp : fe->ident.bs0_exp;
    const int n_ch = fe->ident.n_channels;
    std::memset(unit, 0, sizeof *unit);
    std::memset(floor_y, 0, sizeof(uint16_t) * planes * 65);
    std::memset(residue, 0, sizeof(float) * planes * size_t(slot));
    unit->block_flag = long_block;
    unit->prev_block_flag = uint8_t(fe->prev_block_flag < 0 ? long_block : fe->prev_block_flag);
    for (int ch = 0; ch < SYMGPU_VORBIS_MAX_CHANNELS; ++ch) unit->floor[ch] = 0xffff, unit->do_not_decode[ch] = 1;
    // floors, one per channel (lib.rs:184-207).  A packet that ends inside a floor leaves that floor unused and everything
    // behind it unread -- which the reader reports by failing every later read, exactly the reference's behaviour.
    for (int ch = 0; ch < n_ch; ++ch) {
        const uint8_t floor_idx = mapping.submap_floor[mapping.multiplex[ch]];
        if (uint64_t(floor_base) + floor_idx >= 0xffffu) return SYMGPU_ERR_LIMIT; // unit->floor is 16 bits, 0xffff = unused
        const bool used = read_floor1(*fe, fe->setup.floor1[floor_idx], bs, floor_y + ch * 65);
        unit->do_not_decode[ch] = !used;
        unit->floor[ch] = used ? uint16_t(floor_base + floor_idx) : uint16_t(0xffff);
        if (!used) std::memset(floor_y + ch * 65, 0, sizeof(uint16_t) * 65);
    }
    // non-zero vector propagate (lib.rs:213-225), step by step in mapping order
    for (const auto& cp : mapping.couplings)
        if (unit->do_not_decode[cp.first] != unit->do_not_decode[cp.second]) unit->do_not_decode[cp.first] = unit->do_not_decode[cp.second] = 0;
    // residues, per sub-map (lib.rs:229-248)
    for (int sm = 0; sm < mapping.n_submaps; ++sm) {
        int chans[SYMGPU_VORBIS_MAX_CHANNELS], n_chans = 0;
        for (int ch = 0; ch < n_ch; ++ch)
            if (mapping.multiplex[ch] == sm) chans[n_chans++] = ch;
        const VorbisResidueSetup& r = fe->setup.residues[mapping.submap_residue[sm]];
        if (n_chans == 0) continue;  // (the reference still runs the residue over no channels: nothing is read for types 0 / 1;
                                     //  type 2 divides by the channel count: a malformed setup, refuse it)
        // the partitions must lie inside the vector they are added to
        const size_t n2 = (size_t(1) << bs_exp) >> 1, full = r.type == 2 ? n2 * size_t(n_chans) : n2;
        const size_t begin = std::min<size_t>(r.begin, full), end = std::min<size_t>(r.end, full);
        if (fe->books[r.classbook].dims == 0 || begin + ((end - begin) / r.partition_size) * size_t(r.partition_size) > full) return SYMGPU_ERR_DECODE;
        if (read_residue(*fe, r, bs, bs_exp, chans, n_chans, unit->do_not_decode, residue, slot)) return SYMGPU_ERR_DECODE;
    }
    fe->prev_block_flag = long_block;
    return SYMGPU_OK;
}

// the two record layouts of a decoded packet
constexpr uint32_t planes_of(const symgpu_vorbis_unit*) { return 2; }
symgpu_status decode_into(symgpu_vorbis_fe* fe, const uint8_t* packet, size_t n, uint32_t slot, uint32_t floor_base, uint32_t,
                          symgpu_vorbis_unit* unit, uint16_t* floor_y, float* residue) {
    return symgpu_vorbis_fe_decode(fe, packet, n, slot, floor_base, unit, floor_y, residue);
}
symgpu_status decode_into(symgpu_vorbis_fe* fe, const uint8_t* packet, size_t n, uint32_t slot, uint32_t floor_base, uint32_t planes,
                          symgpu_vorbis_unit_mc* unit, uint16_t* floor_y, float* residue) {
    return symgpu_vorbis_fe_decode_mc(fe, packet, n, slot, floor_base, planes, unit, floor_y, residue);
}
symgpu_status create_for(const symgpu_vorbis_unit*, const uint8_t* ident, size_t n_ident, const uint8_t* setup, size_t n_setup, symgpu_vorbis_fe** out) {
    return symgpu_vorbis_fe_create(ident, n_ident, setup, n_setup, out);
}
symgpu_status create_for(const symgpu_vorbis_unit_mc*, const uint8_t* ident, size_t n_ident, const uint8_t* setup, size_t n_setup, symgpu_vorbis_fe** out) {
    return symgpu_vorbis_fe_create_mc(ident, n_ident, setup, n_setup, out);
}

template <class Unit>
symgpu_status decode_packets(symgpu_vorbis_fe* fe, const uint8_t* data, size_t n, const symgpu_piece* packets, size_t n_packets, uint32_t slot,
                             uint32_t floor_base, uint32_t planes, Unit* units, uint16_t* floor_y, float* residue, uint32_t* packet_of, size_t* n_good) {
    if (!fe || (!data && n) || (n_packets && (!packets || !units || !floor_y || !residue || !packet_of)) || !n_good) return SYMGPU_ERR_ARG;
    if (slot < ((1u << fe->ident.bs1_exp) >> 1)) return SYMGPU_ERR_ARG;
    size_t good = 0;
    for (size_t i = 0; i < n_packets; ++i) {
        if (packets[i].offset > n || packets[i].len > n - packets[i].offset) continue;
        const symgpu_status st = decode_into(fe, data + packets[i].offset, packets[i].len, slot, floor_base, planes, units + good,
                                             floor_y + 65 * size_t(planes) * good, residue + size_t(planes) * slot * good);
        if (st != SYMGPU_OK) continue;  // the caller of the reference drops the packet and goes on
        packet_of[good++] = uint32_t(i);
    }
    *n_good = good;
    return SYMGPU_OK;
}

// A stream's audio packets as independent jobs (DESIGN 10.9): a packet depends on its predecessors only through the previous block
// flag, which is output, not input, of the entropy stage -- the partition-class vector's history never reaches an entry a packet reads
// before writing it, and what a class word writes does not depend on the vector's length beyond the entries it has (the digits kept
// when it is cut are the same most significant ones).  This holds for any number of channels per sub-map: a residue's pass 0 writes the
// class words of every decoded channel of a partition group before any entry of that group is read, a channel only reads its own
// entries [c * parts, (c + 1) * parts), and the vector is at least parts * channels long, so those entries are never cut; what an
// earlier channel's last word spills into them is written in the same packet.  Every thread owns a front-end built from the headers;
// outputs stay at their packet's index (units[i], floor_y[65 planes i], residue[planes slot i]); accepted[0 .. n_good) lists the
// packets the reference decodes, in order, and the previous block flags are chained over exactly those.
template <class Unit>
symgpu_status decode_packets_jobs(const uint8_t* ident, size_t n_ident, const uint8_t* setup, size_t n_setup, const uint8_t* data, size_t n,
                                  const symgpu_piece* packets, size_t n_packets, uint32_t slot, uint32_t floor_base, uint32_t planes, Unit* units,
                                  uint16_t* floor_y, float* residue, uint32_t* accepted, size_t* n_good, uint32_t n_threads) {
    if (n_good) *n_good = 0;
    if ((!data && n) || (n_packets && (!packets || !units || !floor_y || !residue || !accepted)) || !n_good) return SYMGPU_ERR_ARG;
    n_threads = std::max<uint32_t>(1, std::min<uint32_t>({n_threads, 64u, std::max(1u, std::thread::hardware_concurrency()),
                                                           uint32_t(std::min<size_t>(std::max<size_t>(n_packets, 1), 64))}));
    try { // no C++ exception crosses the ABI (vector / thread creation may throw)
    std::vector<symgpu_vorbis_fe*> fes(n_threads, nullptr);
    symgpu_status st = SYMGPU_OK;
    for (uint32_t t = 0; t < n_threads && st == SYMGPU_OK; ++t) st = create_for(units, ident, n_ident, setup, n_setup, &fes[t]);
    if (st == SYMGPU_OK && slot < ((1u << fes[0]->ident.bs1_exp) >> 1)) st = SYMGPU_ERR_ARG;
    if (st == SYMGPU_OK && (planes < fes[0]->ident.n_channels || planes > SYMGPU_VORBIS_MAX_CHANNELS)) st = SYMGPU_ERR_ARG;
    std::vector<uint8_t> ok(n_packets, 0);
    if (st == SYMGPU_OK) {
        std::vector<std::thread> pool;
        for (uint32_t t = 0; t < n_threads; ++t)
            pool.emplace_back([&, t] {
                for (size_t i = t; i < n_packets; i += n_threads) {
                    if (packets[i].offset > n || packets[i].len > n - packets[i].offset) continue;
                    ok[i] = decode_into(fes[t], data + packets[i].offset, packets[i].len, slot, floor_base, planes, units + i,
                                        floor_y + 65 * size_t(planes) * i, residue + size_t(planes) * slot * i) == SYMGPU_OK;
                }
            });
        for (auto& th : pool) th.join();
        size_t good = 0;
        int prev = -1;
        for (size_t i = 0; i < n_packets; ++i) {
            if (!ok[i]) {
                std::memset(units + i, 0, sizeof *units);
                continue;
            }
            units[i].prev_block_flag = uint8_t(prev < 0 ? units[i].block_flag : prev);
            prev = units[i].block_flag;
            accepted[good++] = uint32_t(i);
        }
        *n_good = good;
    }
    for (symgpu_vorbis_fe* fe : fes) symgpu_vorbis_fe_destroy(fe);
    return st;
    } catch (...) {
        *n_good = 0;
        return SYMGPU_ERR_LIMIT;
    }
}

}  // namespace

extern "C" symgpu_status symgpu_vorbis_fe_create(const uint8_t* ident, size_t n_ident, const uint8_t* setup, size_t n_setup, symgpu_vorbis_fe** out) {
    if (!ident || !setup || !out) return SYMGPU_ERR_ARG;
    std::unique_ptr<symgpu_vorbis_fe> fe;
    const symgpu_status st = open_stream(ident, n_ident, setup, n_setup, fe);
    if (st == SYMGPU_OK && !fe->stereo) return SYMGPU_ERR_UNSUPPORTED;  // (more than two channels, or couplings the two-plane record cannot hold)
    if (st != SYMGPU_OK) return st;
    *out = fe.release();
    return SYMGPU_OK;
}
extern "C" symgpu_status symgpu_vorbis_fe_create_mc(const uint8_t* ident, size_t n_ident, const uint8_t* setup, size_t n_setup, symgpu_vorbis_fe** out) {
    if (!ident || !setup || !out) return SYMGPU_ERR_ARG;
    std::unique_ptr<symgpu_vorbis_fe> fe;
    const symgpu_status st = open_stream(ident, n_ident, setup, n_setup, fe);
    if (st != SYMGPU_OK) return st;
    *out = fe.release();
    return SYMGPU_OK;
}
extern "C" void symgpu_vorbis_fe_destroy(symgpu_vorbis_fe* fe) { delete fe; }
extern "C" void symgpu_vorbis_fe_reset(symgpu_vorbis_fe* fe) {
    if (fe) fe->prev_block_flag = -1;
}

extern "C" symgpu_status symgpu_vorbis_fe_config(const symgpu_vorbis_fe* fe, symgpu_vorbis_stream* stream, symgpu_vorbis_floor1* floors, uint32_t* n_floors) {
    if (!fe || !stream || !floors || !n_floors || !fe->stereo) return SYMGPU_ERR_ARG;
    *stream = symgpu_vorbis_stream{fe->ident.bs0_exp, fe->ident.bs1_exp, fe->ident.n_channels,
                                   uint8_t(fe->setup.mappings[fe->setup.modes[0].second].couplings.empty() ? 0 : 1)};
    floor_records(fe, floors, n_floors);
    return SYMGPU_OK;
}
extern "C" symgpu_status symgpu_vorbis_fe_config_mc(const symgpu_vorbis_fe* fe, symgpu_vorbis_stream_mc* stream, symgpu_vorbis_floor1* floors, uint32_t* n_floors) {
    if (!fe || !stream || !floors || !n_floors) return SYMGPU_ERR_ARG;
    std::memset(stream, 0, sizeof *stream);
    stream->bs0_exp = fe->ident.bs0_exp, stream->bs1_exp = fe->ident.bs1_exp, stream->channels = fe->ident.n_channels;
    const auto& couplings = fe->setup.mappings[fe->setup.modes[0].second].couplings;
    stream->n_couplings = uint8_t(couplings.size());
    for (size_t k = 0; k < couplings.size(); ++k) stream->magnitude_ch[k] = couplings[k].first, stream->angle_ch[k] = couplings[k].second;
    floor_records(fe, floors, n_floors);
    return SYMGPU_OK;
}

extern "C" symgpu_status symgpu_vorbis_fe_decode(symgpu_vorbis_fe* fe, const uint8_t* packet, size_t n, uint32_t slot, uint32_t floor_base,
                                                 symgpu_vorbis_unit* unit, uint16_t* floor_y, float* residue) {
    if (!fe || (!packet && n) || !unit || !floor_y || !residue || !fe->stereo) return SYMGPU_ERR_ARG;
    if (slot < ((1u << fe->ident.bs1_exp) >> 1)) return SYMGPU_ERR_ARG;
    symgpu_vorbis_unit_mc u;
    const symgpu_status st = decode_packet(fe, packet, n, slot, floor_base, 2, &u, floor_y, residue);
    if (st != SYMGPU_OK) return st;
    std::memset(unit, 0, sizeof *unit);
    unit->block_flag = u.block_flag, unit->prev_block_flag = u.prev_block_flag;
    for (int c = 0; c < 2; ++c) unit->do_not_decode[c] = u.do_not_decode[c], unit->floor[c] = u.floor[c];
    return SYMGPU_OK;
}
extern "C" symgpu_status symgpu_vorbis_fe_decode_mc(symgpu_vorbis_fe* fe, const uint8_t* packet, size_t n, uint32_t slot, uint32_t floor_base,
                                                    uint32_t planes, symgpu_vorbis_unit_mc* unit, uint16_t* floor_y, float* residue) {
    if (!fe || (!packet && n) || !unit || !floor_y || !residue) return SYMGPU_ERR_ARG;
    if (slot < ((1u << fe->ident.bs1_exp) >> 1) || planes < fe->ident.n_channels || planes > SYMGPU_VORBIS_MAX_CHANNELS) return SYMGPU_ERR_ARG;
    return decode_packet(fe, packet, n, slot, floor_base, planes, unit, floor_y, residue);
}

extern "C" symgpu_status symgpu_vorbis_fe_decode_packets(symgpu_vorbis_fe* fe, const uint8_t* data, size_t n, const symgpu_piece* packets, size_t n_packets,
                                                         uint32_t slot, uint32_t floor_base, symgpu_vorbis_unit* units, uint16_t* floor_y, float* residue,
                                                         uint32_t* packet_of, size_t* n_good) {
    if (fe && !fe->stereo) return SYMGPU_ERR_ARG;
    return decode_packets(fe, data, n, packets, n_packets, slot, floor_base, 2, units, floor_y, residue, packet_of, n_good);
}
extern "C" symgpu_status symgpu_vorbis_fe_decode_packets_mc(symgpu_vorbis_fe* fe, const uint8_t* data, size_t n, const symgpu_piece* packets,
                                                            size_t n_packets, uint32_t slot, uint32_t floor_base, uint32_t planes,
                                                            symgpu_vorbis_unit_mc* units, uint16_t* floor_y, float* residue, uint32_t* packet_of,
                                                            size_t* n_good) {
    if (fe && (planes < fe->ident.n_channels || planes > SYMGPU_VORBIS_MAX_CHANNELS)) return SYMGPU_ERR_ARG;
    return decode_packets(fe, data, n, packets, n_packets, slot, floor_base, planes, units, floor_y, residue, packet_of, n_good);
}

extern "C" symgpu_status symgpu_vorbis_fe_decode_packets_jobs(const uint8_t* ident, size_t n_ident, const uint8_t* setup, size_t n_setup, const uint8_t* data,
                                                              size_t n, const symgpu_piece* packets, size_t n_packets, uint32_t slot, uint32_t floor_base,
                                                              symgpu_vorbis_unit* units, uint16_t* floor_y, float* residue, uint32_t* accepted, size_t* n_good,
                                                              uint32_t n_threads) {
    return decode_packets_jobs(ident, n_ident, setup, n_setup, data, n, packets, n_packets, slot, floor_base, 2, units, floor_y, residue, accepted,
                               n_good, n_threads);
}
extern "C" symgpu_status symgpu_vorbis_fe_decode_packets_jobs_mc(const uint8_t* ident, size_t n_ident, const uint8_t* setup, size_t n_setup,
                                                                 const uint8_t* data, size_t n, const symgpu_piece* packets, size_t n_packets,
                                                                 uint32_t slot, uint32_t floor_base, uint32_t planes, symgpu_vorbis_unit_mc* units,
                                                                 uint16_t* floor_y, float* residue, uint32_t* accepted, size_t* n_good,
                                                                 uint32_t n_threads) {
    return decode_packets_jobs(ident, n_ident, setup, n_setup, data, n, packets, n_packets, slot, floor_base, planes, units, floor_y, residue,
                               accepted, n_good, n_threads);
}

// lib.rs:771-788 (Vorbis I 4.3.9): the output plane of Vorbis channel i
extern "C" symgpu_status symgpu_vorbis_channel_map(uint32_t channels, uint8_t* plane_of_channel) {
    static const uint8_t maps[SYMGPU_VORBIS_MAX_CHANNELS][SYMGPU_VORBIS_MAX_CHANNELS] = {
        {0}, {0, 1}, {0, 2, 1}, {0, 1, 2, 3}, {0, 2, 1, 3, 4}, {0, 2, 1, 4, 5, 3}, {0, 2, 1, 5, 6, 4, 3}, {0, 2, 1, 6, 7, 4, 5, 3},
    };
    if (!plane_of_channel || channels < 1 || channels > SYMGPU_VORBIS_MAX_CHANNELS) return SYMGPU_ERR_ARG;
    std::memcpy(plane_of_channel, maps[channels - 1], channels);
    return SYMGPU_OK;
}
