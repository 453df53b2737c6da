// Function-level differential test of include/rans_byte.h, rans64.h, rans_word_sse41.h against the reference's headers.
// body.inc drives every function of the three APIs and records everything observable; this harness prints one digest
// line per API and seed.  tests/test_header_parity.py builds it against include/*.h and requires the lines the same
// harness printed when built against the reference's own headers (-DRANS_REF_HEADERS, REFDIR replaced by the
// reference checkout's path), which tests/golden/make_reference_vectors.py stored in tests/golden/reference_vectors.json.
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <stdio.h>
#include <assert.h>
#include <smmintrin.h>
#include <algorithm>
#include <random>
#include <vector>

#ifdef RANS_REF_HEADERS
#include "REFDIR/platform.h"
#include "REFDIR/rans_byte.h"
#include "REFDIR/rans64.h"
#include "REFDIR/rans_word_sse41.h"
#else
#include "platform.h"
#include "rans_byte.h"
#include "rans64.h"
#include "rans_word_sse41.h"
#endif
#include "body.inc"

// FNV-1a, 64 bit: one digest over the recorded values, one over the produced stream bytes
static uint64_t fnv1a(const void* p, size_t n)
{
    const uint8_t* q = (const uint8_t*)p;
    uint64_t h = 0xcbf29ce484222325ull;
    for (size_t i = 0; i < n; i++) h = (h ^ q[i]) * 0x100000001b3ull;
    return h;
}

static void report(const char* what, uint64_t seed, const Out& o)
{
    printf("%s seed %llu: round trips %d, %zu values fnv1a %016llx, %zu stream bytes fnv1a %016llx\n", what,
           (unsigned long long)seed, (int)o.round_trips, o.vals.size(),
           (unsigned long long)fnv1a(o.vals.data(), o.vals.size() * sizeof(uint64_t)), o.bytes.size(),
           (unsigned long long)fnv1a(o.bytes.data(), o.bytes.size()));
}

int main()
{
    for (uint64_t seed = 1; seed <= 3; seed++) {
        { Out o; run_byte(seed, o); report("rans_byte.h", seed, o); }
        { Out o; run_64(seed, o); report("rans64.h", seed, o); }
        { Out o; run_word(seed, o); report("rans_word_sse41.h", seed, o); }
    }
    return 0;
}
