// Chunked long-row sweep (pg_sweep_long.cuh) for P planes, built with -DPG_P=<planes> so the two
// plane counts compile in parallel: P = 5 with W = 64..1024, P = 8 with W = 16..1024 (multiples of 8).
#include "pg_sweep_long.cuh"

#ifndef PG_P
#error "compile with -DPG_P=<planes>"
#endif

#define PG_CAT2(a, b) a##b
#define PG_NAME(P) PG_CAT2(sweep_wide_p, P)

namespace pg {
int PG_NAME(PG_P)(const SweepParams& prm, const SweepLaunch& l, int words) { return launch_long<PG_P, true>(prm, l, words); }
}  // namespace pg
