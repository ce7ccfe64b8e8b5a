// scan_hwa_host.cpp - TEST INFRASTRUCTURE: the HWA division of k_scan's 8-bit accumulator lanes (hdp_b200/csrc/metric.cu, flush:
// (f * scan_hwa_rcp(nn)) >> 16 in 32-bit unsigned arithmetic) against trunc(f / nn) for every pair the lanes can hold.  Not part of
// the product.
//     g++ -O2 -shared -fPIC -I hdp_b200/csrc tests/scan_hwa_host.cpp -o <tmp>/libscan_hwa_host.so
#include <stdint.h>

#include "seams.h"

extern "C" {

// Number of pairs f, nn in [0, 256) where the kernel's form differs from nn ? f / nn : 0; the first such pair goes to bad[0..1].
int64_t scan_hwa_mismatches(uint32_t *bad)
{
    int64_t n = 0;
    for (uint32_t nn = 0; nn < 256; nn++)
        for (uint32_t f = 0; f < 256; f++) {
            const uint32_t got = (f * hdp::scan_hwa_rcp(nn)) >> 16, want = nn ? f / nn : 0u;
            if (got != want && n++ == 0) { bad[0] = f; bad[1] = nn; }
        }
    return n;
}

}  // extern "C"
