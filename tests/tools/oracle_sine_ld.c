/*
 * oracle_sine_ld.c — oracle_sine.c compiled in x87 80-bit arithmetic (TEST INFRASTRUCTURE ONLY): orc_approx_logl_sine_grad_batch_ld,
 * for telling conditioning from error in comparisons with the sinusoidal-mean entries.
 */
#define ORC_GRAD_LONG_DOUBLE 1
#include "oracle_sine.c"
