// Sharded particle system of TemperedLikelihoodSMC (SURVEY 8(e), north_star item 4).
//
// One process per GPU; rank r owns the contiguous particle range [lo(r), lo(r) + n(r)).  The ranks
// never call a host-side collective per temperature: they talk through peer-accessible device memory
// (NVLink P2P / symmetric memory) --
//   * small fixed-size MESSAGES posted into every rank's mailbox (payload, then a release store of the
//     step number; the reader spins with acquire loads): local max of the log-weights, local
//     fixed-point weight mass, "my resample indices are final";
//   * the resample INDICES a rank resolves for points that land in its own CDF interval, stored straight
//     into the idx array of the rank that owns the slot;
//   * the particle ROWS, read from their owner's array by the next move kernel.
// With world == 1 the same kernels run; every wait is already satisfied by stream order.
//
// The device side of the protocol (geometry, mailbox layout, waits and posts) lives in smc_mailbox.cuh, which the
// SMC kernels of runtime-compiled user models share.
#pragma once
#include "common.cuh"
#include "smc_mailbox.cuh"
