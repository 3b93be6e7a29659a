/*
 * psa_internal.h -- test and measurement hooks of libpsa.so.  NOT part of the drop-in ABI
 * (include/psa.h): nothing the reference's callers need lives here.  tests/, bench.py and tools/
 * use it to select a kernel variant or to time one kernel of a step on its own; the shipped
 * behaviour is every option at its default, and no launch path reads the environment.
 */
#ifndef PSA_INTERNAL_H
#define PSA_INTERNAL_H

#include "../../include/psa.h"

#ifdef __cplusplus
extern "C" {
#endif

/* name: pack, pipeline, pack_traceback, pack_skip_walk, pack_ctas_per_sm, pack_chunk, pack_serial_fills, pack_long_k,
 *       long_geometry, long_ctas_per_sm, long_band, long_tb_chunk, long_systolic, systolic_warps_per_sm, systolic_kc,
 *       systolic_rb, timing
 * (struct psa_options in psa_common.cuh).  Returns PSA_ERR_ARG for an unknown name. */
int psa_ctx_set_option(psa_ctx* ctx, const char* name, long long value);

#ifdef __cplusplus
}
#endif
#endif
