// scan_onset_host.cpp - TEST INFRASTRUCTURE: the packed HWO / HWE update of k_scan's ONSET accumulators (hdp_b200/csrc/seams.h:
// scan_onset_update, called per accumulator register from metric.cu's account) against a lane-by-lane model, for both lane widths.
// Not part of the product.
//     g++ -O2 -shared -fPIC -I hdp_b200/csrc tests/scan_onset_host.cpp -o <tmp>/libscan_onset_host.so
#include <stdint.h>
#include <initializer_list>

#include "seams.h"

extern "C" {

// Every selection of lanes (sel, and first within sel: first lanes have no block yet, so their onset lane holds 0), every prior lane
// value from {0, 1, max - 1, max} (the others' onset and end lanes), and every offset a lane holds (lo, last in [0, max]; max = 254
// for 8-bit lanes, whose seasons have at most 255 days, 65534 for 16-bit lanes).  The onset and end updates use one offset each and
// do not touch each other's register, so the two offsets are swept one at a time (the other one at 0 and at max).  Returns the
// number of mismatching cases; the first one goes to bad[0..5] = {bits, sel, first, lo, last, prior pattern}.
int64_t scan_onset_mismatches(int bits, uint32_t *bad)
{
    const int per = 32 / bits;
    const uint32_t lane_mask = bits == 8 ? 0xffu : 0xffffu, vmax = bits == 8 ? 254u : 65534u;
    const uint32_t prior_vals[4] = {0u, 1u, vmax - 1u, vmax};
    int n_prior = 1;
    for (int h = 0; h < per; h++) n_prior *= 4;
    int64_t n = 0;
    for (uint32_t sel = 0; sel < (1u << per); sel++)
        for (uint32_t first = sel;; first = (first - 1u) & sel) {                 // every subset of sel
            for (int pat = 0; pat < n_prior; pat++) {
                uint32_t ons0 = 0u, end0 = 0u, sel_s = 0u, first_s = 0u;
                for (int h = 0, q = pat; h < per; h++, q /= 4) {
                    const uint32_t v = prior_vals[q % 4], w = prior_vals[(q / 2 + h) % 4];
                    ons0 |= ((first >> h) & 1u ? 0u : v) << (bits * h);
                    end0 |= w << (bits * h);
                    sel_s |= ((sel >> h) & 1u) << (bits * h);
                    first_s |= ((first >> h) & 1u) << (bits * h);
                }
                for (int sweep = 0; sweep < 4; sweep++)
                    for (uint32_t v = 0; v <= vmax; v++) {
                        const uint32_t fixed = (sweep & 2) ? vmax : 0u;
                        const uint32_t lo = (sweep & 1) ? fixed : v, last = (sweep & 1) ? v : fixed;
                        uint32_t ons = ons0, end = end0;
                        hdp::scan_onset_update(ons, end, first_s, sel_s, lo, last, lane_mask);
                        bool ok = true;
                        for (int h = 0; h < per; h++) {
                            const uint32_t o0 = (ons0 >> (bits * h)) & lane_mask, e0 = (end0 >> (bits * h)) & lane_mask;
                            const uint32_t want_o = (first >> h) & 1u ? lo : o0, want_e = (sel >> h) & 1u ? last : e0;
                            ok = ok && ((ons >> (bits * h)) & lane_mask) == want_o && ((end >> (bits * h)) & lane_mask) == want_e;
                        }
                        if (!ok && n++ == 0) {
                            bad[0] = (uint32_t)bits; bad[1] = sel; bad[2] = first; bad[3] = lo; bad[4] = last; bad[5] = (uint32_t)pat;
                        }
                    }
            }
            if (first == 0u) break;
        }
    return n;
}

// HWO / HWE as the flush stores them: the lane's value, 0xFFFF where HWF = 0
int64_t scan_onset_value_mismatches(void)
{
    int64_t n = 0;
    for (uint32_t f = 0; f < 65536; f += 1)
        for (uint32_t v : {0u, 1u, 254u, 65534u}) n += hdp::scan_onset_value(f, v) != (f ? v : 0xffffu);
    return n;
}

}  // extern "C"
