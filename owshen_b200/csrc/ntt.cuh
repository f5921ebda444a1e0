// owshen_b200/csrc/ntt.cuh -- interface of the batched NTT module.
#pragma once
#include "common.cuh"

namespace og {
// `batch` contiguous transforms of 2^log_n Montgomery-form elements, in place; tmp: batch*n scratch
// (only touched when log_n > 10).
// fold: 0 = a complete transform.  An inverse transform followed by a forward coset transform of the same data (the prover's
// a, b, c) can leave the 1/n to the coset factors of the second one: fold = 1 on the inverse (plain, non-coset) call, fold = 2 on
// the forward coset call -- one product per element fewer for the pair.
int32_t ntt_mont_dev(og_ctx* ctx, Fr* data, Fr* tmp, uint32_t log_n, uint32_t batch, int inverse, int coset, int fold = 0);
void ntt_free_tables(og_ctx* ctx);
}  // namespace og
