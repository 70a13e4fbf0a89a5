// Deterministic one-pass field reductions (min, max, sum, sum of squares) over a box of 1-4 strided allocations: the
// filters of the reference's astaroth extract (astaroth/reductions.cuh:18-52, RTYPE_* of astaroth/user_defines.h:161-169)
// evaluated and accumulated in FP64.  Bandwidth-bound: no tensor cores.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace sb {

enum ReduceKind { kReduceValue = 0, kReduceDiff = 1, kReduceVector = 2, kReduceExp = 3, kReduceAlfven = 4 };

// operand count of each kind
int reduce_num_operands(int kind);

// Workspace layout (caller-owned device memory, zeroed once): the result {min, max, sum, sum2} (4 doubles) at byte 0,
// the uint32 ticket of the last-CTA combine at byte 32, the CTA partials (4 doubles per CTA) from byte 64.
int64_t reduce_workspace_bytes(int num_sms);

// One launch over the ALLOCATION-relative box [lo, hi) of every operand (same pitch and slice).  Returns the number of
// launches issued (always 1: an empty box still writes the identities).
int launch_reduce(int kind, const char *const ops[4], int dtype_size, long long pitch, long long slice, const int lo[3],
                  const int hi[3], void *workspace, int num_sms, cudaStream_t stream);

} // namespace sb
