// Long-row sweep (pg_sweep_long.cuh) with whole stream rows in the ring: P = 5, W = 24..56.
#include "pg_sweep_long.cuh"

namespace pg {

// planes = 5 only (protein alphabets); words = 24..56, a multiple of 8
int sweep_long_p5(const SweepParams& prm, const SweepLaunch& l, int words) { return launch_long<5, false>(prm, l, words); }

}  // namespace pg
