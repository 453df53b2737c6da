// Differential test of include/rans_alias.h against the reference's own alias code, which lives in its driver
// (main_alias.cpp: SymbolStats::make_alias_table, RansEncPutAlias, RansDecGetAlias).  For every seed and scale_bits the
// harness prints one digest line over everything observable: the alias tables, the encoder state after every symbol,
// the stream, and the decoder's symbol, state and cursor after every step.
//
// Built with -DRANS_REF_DRIVER (REFDIR replaced by the reference checkout's path), the model, tables and steps come from
// main_alias.cpp, #included where it lies (its main renamed; nothing is copied), and our functions are driven beside
// them on the driver's own SymbolStats and on RansAliasTables: any difference fails the run.  That build also prints
// each model's frequencies ("freqs ..." lines).  Built without it, the harness reads those frequencies from stdin and
// runs include/rans_alias.h alone; tests/test_header_parity.py requires its digest lines to be the ones the driver
// build printed (tests/golden/reference_vectors.json).
// system headers first, outside the namespaces: their include guards then make the driver's own #includes no-ops
#include <stdio.h>
#include <stdarg.h>
#include <stdlib.h>
#include <stdint.h>
#include <string.h>
#include <assert.h>
#include <time.h>
#ifndef __STDC_FORMAT_MACROS
#define __STDC_FORMAT_MACROS
#endif
#include <inttypes.h>
#include <x86intrin.h>

#include <new>
#include <random>
#include <vector>

#ifdef RANS_REF_DRIVER
namespace ref {
#define main ref_driver_main_alias
#include "REFDIR/main_alias.cpp"
#undef main
}
#undef RANS_BYTE_HEADER
#undef RansAssert
#undef RANS_BYTE_L
#endif
namespace ours {
#include "rans_alias.h"
}

struct Fnv1a {                                     // 64-bit FNV-1a over everything added
    uint64_t h = 0xcbf29ce484222325ull;
    void add(const void* p, size_t n) { const uint8_t* q = (const uint8_t*)p; for (size_t i = 0; i < n; i++) h = (h ^ q[i]) * 0x100000001b3ull; }
};

struct Trace {
    std::vector<uint32_t> enc;                     // encoder state after each symbol (input order)
    std::vector<uint8_t> stream;
    std::vector<uint32_t> dec;                     // per step: symbol, state, cursor offset
    bool round_trips = true;
    bool operator==(const Trace& o) const { return enc == o.enc && stream == o.stream && dec == o.dec && round_trips == o.round_trips; }
};

// one encode + decode of `in` with coder C's step functions on table object `tab`
template <class C, class Tab> static Trace trace(Tab* tab, const std::vector<uint8_t>& in, uint32_t scale_bits)
{
    Trace tr;
    const size_t n = in.size(), cap = 2 * n + 64;
    std::vector<uint8_t> buf(cap);
    uint8_t* p = buf.data() + cap;
    typename C::State x;
    C::EncInit(&x);
    tr.enc.resize(n);
    for (size_t i = n; i-- > 0;) {
        C::EncPut(&x, &p, tab, in[i], scale_bits);
        tr.enc[i] = x;
    }
    C::EncFlush(&x, &p);
    tr.stream.assign(p, buf.data() + cap);
    uint8_t* q = p;
    C::DecInit(&x, &q);
    for (size_t i = 0; i < n; i++) {
        const uint32_t s = C::DecGet(&x, tab, scale_bits);
        C::DecRenorm(&x, &q);
        tr.round_trips &= s == in[i];
        tr.dec.push_back(s); tr.dec.push_back(x); tr.dec.push_back((uint32_t)(q - p));
    }
    return tr;
}

struct Ours {
    typedef ours::RansState State;
    static void EncInit(State* x) { ours::RansEncInit(x); }
    template <class T> static void EncPut(State* x, uint8_t** p, T* t, int s, uint32_t sb) { ours::RansEncPutAlias(x, p, t, s, sb); }
    static void EncFlush(State* x, uint8_t** p) { ours::RansEncFlush(x, p); }
    static void DecInit(State* x, uint8_t** p) { ours::RansDecInit(x, p); }
    template <class T> static uint32_t DecGet(State* x, T* t, uint32_t sb) { return ours::RansDecGetAlias(x, t, sb); }
    static void DecRenorm(State* x, uint8_t** p) { ours::RansDecRenorm(x, p); }
};

#ifdef RANS_REF_DRIVER
struct Ref {
    typedef ref::RansState State;
    static void EncInit(State* x) { ref::RansEncInit(x); }
    static void EncPut(State* x, uint8_t** p, ref::SymbolStats* t, int s, uint32_t sb) { ref::RansEncPutAlias(x, p, t, s, sb); }
    static void EncFlush(State* x, uint8_t** p) { ref::RansEncFlush(x, p); }
    static void DecInit(State* x, uint8_t** p) { ref::RansDecInit(x, p); }
    static uint32_t DecGet(State* x, ref::SymbolStats* t, uint32_t sb) { return ref::RansDecGetAlias(x, t, sb); }
    static void DecRenorm(State* x, uint8_t** p) { ref::RansDecRenorm(x, p); }
};
#endif

static uint64_t table_digest(const uint32_t* divider, const uint32_t* slot_adjust, const uint32_t* slot_freqs, const uint8_t* sym_id,
                             const uint32_t* remap, size_t remap_len)
{
    Fnv1a d;
    d.add(divider, 256 * 4); d.add(slot_adjust, 512 * 4); d.add(slot_freqs, 512 * 4); d.add(sym_id, 512); d.add(remap, remap_len * 4);
    return d.h;
}

static int run(uint64_t seed, uint32_t scale_bits, size_t n)
{
    std::mt19937_64 rng(seed);
    std::vector<uint8_t> in(n);
    for (size_t i = 0; i < n; i++) {
        const uint64_t r = rng();
        in[i] = (uint8_t)((r & 0xff) & ((r >> 8) & 0xff) & (seed % 3 ? 0xff : (r >> 16) & 0xff));      // skewed
    }
    ours::RansAliasTables t;
#ifdef RANS_REF_DRIVER
    ref::SymbolStats st;
    st.count_freqs(in.data(), n);
    st.normalize_freqs(1u << scale_bits);
    st.make_alias_table();
    memcpy(t.freqs, st.freqs, sizeof t.freqs);
    memcpy(t.cum_freqs, st.cum_freqs, sizeof t.cum_freqs);
    printf("freqs seed %llu scale_bits %u:", (unsigned long long)seed, scale_bits);
    for (int s = 0; s < 256; s++) printf(" %u", st.freqs[s]);
    printf("\n");
#else
    t.cum_freqs[0] = 0;
    for (int s = 0; s < 256; s++) {
        if (scanf("%u", &t.freqs[s]) != 1) { printf("missing frequencies (seed %llu, scale_bits %u)\n", (unsigned long long)seed, scale_bits); return 1; }
        t.cum_freqs[s + 1] = t.cum_freqs[s] + t.freqs[s];
    }
#endif
    std::vector<uint32_t> remap(t.cum_freqs[256]);
    t.alias_remap = remap.data();
    if (ours::RansAliasTablesInit(&t) != 0) { printf("RansAliasTablesInit failed\n"); return 1; }
    const uint64_t tables = table_digest(t.divider, t.slot_adjust, t.slot_freqs, t.sym_id, remap.data(), remap.size());
    Trace tr = trace<Ours>(&t, in, scale_bits);
#ifdef RANS_REF_DRIVER
    if (tables != table_digest(st.divider, st.slot_adjust, st.slot_freqs, st.sym_id, st.alias_remap, st.cum_freqs[256]) ||
        memcmp(remap.data(), st.alias_remap, remap.size() * sizeof(uint32_t))) {
        printf("alias tables differ (seed %llu, scale_bits %u)\n", (unsigned long long)seed, scale_bits);
        return 1;
    }
    const Trace want = trace<Ref>(&st, in, scale_bits);
    if (!(trace<Ours>(&st, in, scale_bits) == want) || !(tr == want)) {   // ours on the driver's struct and on ours
        printf("encoder, stream or decoder differs (seed %llu, scale_bits %u)\n", (unsigned long long)seed, scale_bits);
        return 1;
    }
#endif
    Fnv1a e, s, d;
    e.add(tr.enc.data(), tr.enc.size() * 4); s.add(tr.stream.data(), tr.stream.size()); d.add(tr.dec.data(), tr.dec.size() * 4);
    printf("seed %llu scale_bits %u: %zu symbols, round trips %d, tables fnv1a %016llx, encoder fnv1a %016llx, "
           "%zu stream bytes fnv1a %016llx, decoder fnv1a %016llx\n", (unsigned long long)seed, scale_bits, n, (int)tr.round_trips,
           (unsigned long long)tables, (unsigned long long)e.h, tr.stream.size(), (unsigned long long)s.h, (unsigned long long)d.h);
    return 0;
}

int main()
{
    int bad = 0;
    for (uint64_t seed = 1; seed <= 4; seed++)
        for (uint32_t sb : {8u, 11u, 14u, 16u}) bad += run(seed, sb, 20000 + 997 * seed);
    return bad;
}
