/*
 * mmbo_substructure.h — CPU restatement (plain C) of mmb_jet_substructure (include/mmbridge.h).
 *
 * TEST INFRASTRUCTURE ONLY, like oracle/: nothing in the product path links or calls it; the tests and
 * tools/substructure_bench.py use it as the checker and as the CPU context of the measured rate.  It lives beside
 * oracle/ rather than inside it so that the pinned generation oracle stays byte for byte what its fixtures check.
 *
 * The signature mirrors the C ABI (host pointers here, device pointers there).
 */
#ifndef MMBO_SUBSTRUCTURE_H
#define MMBO_SUBSTRUCTURE_H

#include "../include/mmbridge.h"

#ifdef __cplusplus
extern "C" {
#endif

void mmbo_jet_substructure(const float* x, const uint8_t* mask, const float* mean, const float* sd, int B, int N, float R, float beta,
                           float* out, int16_t* axes);
int mmbo_substructure_threads(void);

#ifdef __cplusplus
}
#endif
#endif /* MMBO_SUBSTRUCTURE_H */
