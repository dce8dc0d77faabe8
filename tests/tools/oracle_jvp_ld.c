/*
 * oracle_jvp_ld.c — oracle_jvp.c compiled in x87 80-bit arithmetic (TEST INFRASTRUCTURE ONLY): orc_celerite_logl_jvp_batch_ld and
 * orc_approx_features_logl_grad_batch_ld, for telling conditioning from error in derivative comparisons.
 */
#define ORC_JVP_LONG_DOUBLE 1
#include "oracle_jvp.c"
