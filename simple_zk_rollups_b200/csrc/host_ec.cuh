// Host-side curve checks and pairings (verify.cu) on points in the binary key encoding: affine, Fq-M,
// x == 0 marks infinity.  Used by the setup ceremony (ceremony.cu) to validate inputs before any launch and to
// check phase-2 contributions.
#pragma once
#include <cstdint>

namespace zkr {

enum PointCheck { PT_OK = 0, PT_INFINITY, PT_RANGE, PT_OFF_CURVE, PT_SUBGROUP };
// group 1: 64 B, group 2: 128 B (x.c0|x.c1|y.c0|y.c1).  PT_INFINITY if x == 0, else PT_RANGE if a coordinate is >= q,
// PT_OFF_CURVE, and for G2 with `subgroup` PT_SUBGROUP outside the order-r subgroup.
int host_point_check(int group, const void* mont, bool subgroup);
// prod_i e(+-P_i, Q_i) == 1 for n <= 8 pairs of points that pass host_point_check (P_i negated where negate[i])
bool host_pairing_is_one(const void* const* g1_mont, const bool* negate, const void* const* g2_mont, int n);
// a zkr_msm result (std form, all-zero = infinity) in the key encoding; false if a coordinate is >= q
bool host_g1_std_to_mont(const void* std64, void* mont64);

}  // namespace zkr
