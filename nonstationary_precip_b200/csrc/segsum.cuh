// Shared by the pair-sum kernels (gibbs_segsum.cu) and their plan-level caller (svgp_step.cu).
#pragma once

namespace npgp {

// The pair-sum workspace begins with an int that the scan kernel sets to 1 when seg is not non-decreasing from 0 to n (the
// outputs are then NaN); callers that add further terms read it to fill theirs with NaN as well.
inline const int* segsum_bad_flag(const void* work) { return static_cast<const int*>(work); }

}  // namespace npgp
