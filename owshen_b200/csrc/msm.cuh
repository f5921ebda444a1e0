// owshen_b200/csrc/msm.cuh -- interface of the bucket-method (Pippenger) MSM engine shared by the
// one-shot MSM entry points (og_msm_g1/g2) and the batched Groth16 prover.
#pragma once
#include "common.cuh"

namespace og {

// How scalars are cut into signed c-bit digits and where each (digit, point) pair goes.
//   key   = (problem * key_stride_problem + window * key_stride_window) * nb + (|digit| - 1)
//   entry = ((index + window * tidx_window_stride) << 1) | (digit < 0)
// One-shot MSM:   groups are windows  (key_stride_problem = 0, key_stride_window = 1, tidx stride 0).
// Batched prover: groups are proofs   (key_stride_problem = 1, key_stride_window = 0) and the table
//                 holds the precomputed multiples 2^(c*w) * P_i at index i + w * n_points.
struct DigitPlan {
    const uint32_t* scalars;     // 8 x u32 per scalar; canonical integers or Montgomery Fr
    uint64_t n;                  // scalars per problem
    uint64_t scalar_stride;      // elements between consecutive problems
    uint32_t n_problems;
    uint32_t c, n_windows, nb;   // nb = 2^(c-1) buckets per group
    uint32_t key_stride_problem, key_stride_window;
    uint32_t tidx_window_stride;
    int32_t montgomery;          // 1: scalars are Montgomery-form Fr and are converted on the fly
};

static inline uint32_t msm_windows(uint32_t c) { return (255 + c - 1) / c; }

// The digit sort (msm_sort.cu; the same for both curves).
// counts[n_keys] must be zero on entry; fills counts, offsets (exclusive scan), sorted entries.
// Returns total number of entries through *d_total (device pointer inside offsets[n_keys]).
int32_t msm_sort_digits(og_ctx* ctx, const DigitPlan& plan, uint32_t n_keys, uint32_t* d_counts,
                        uint32_t* d_offsets /* n_keys + 1 */, uint32_t* d_cursor, uint32_t* d_sorted);

// The engine is one set of templates over the coordinate field F: Fq for G1, Fq2 for G2.  msm.cu defines them and is
// compiled once per field; each of its two objects instantiates every template below for its own field.

// Accumulate every bucket and reduce each group to sum_b (b+1) * bucket_b.
// d_buckets: n_groups * nb XYZZ scratch; d_lvl: msm_lvl_elems(n_groups, nb) XYZZ scratch;
// d_heavy: 2 * n_keys + 4 u32 scratch; n_entries_max: upper bound on the sorted entries (sets the heavy-bucket cap);
// d_perm: n_keys u32 scratch (the sort's cursor array may be reused); result: d_totals[n_groups].
// few_groups (one-shot MSMs, groups = windows): the levels above the first are reduced as tree sums.
template <class F>
int32_t msm_buckets(og_ctx* ctx, const Affine<F>* d_table, const uint32_t* d_sorted, const uint32_t* d_offsets,
                    const uint32_t* d_counts, uint32_t n_groups, uint32_t nb, uint64_t n_entries_max, XYZZ<F>* d_buckets,
                    XYZZ<F>* d_lvl, uint32_t* d_heavy, uint32_t* d_perm, XYZZ<F>* d_totals, bool few_groups = false);
static inline size_t msm_lvl_elems(uint32_t n_groups, uint32_t nb) { return 4 * ((size_t)n_groups * ((nb + 7) / 8) + 16); }   // RED_FAN = 8

// one-shot MSM on device buffers holding boundary bytes (affine points, canonical scalars); d_out: one point
template <class F> int32_t msm_dev(og_ctx* ctx, const uint8_t* d_points, const uint8_t* d_scalars, uint64_t n, uint8_t* d_out);
// plain sum of n points in boundary bytes
template <class F> int32_t sum_points_dev(og_ctx* ctx, const uint8_t* d_points, uint64_t n, uint8_t* d_out);

// boundary conversions for points
template <class F> int32_t points_to_mont(og_ctx* ctx, const uint8_t* d_in, uint64_t n, Affine<F>* d_out);
template <class F> int32_t points_to_bytes(og_ctx* ctx, const Affine<F>* d_in, uint64_t n, uint8_t* d_out);

// fixed-base window tables: table[w * n + i] = 2^(c*w) * P_i  (w < n_windows), affine Montgomery.
// table[0..n) must already hold the points.
template <class F> int32_t build_table(og_ctx* ctx, Affine<F>* d_table, uint32_t n, uint32_t c, uint32_t n_windows);

// out[i] = scalars[i] * generator of G1 / G2 (setup): scalars canonical bytes on device, out affine Montgomery
template <class F> int32_t fixed_base_mul(og_ctx* ctx, const uint8_t* d_scalars, uint64_t n, Affine<F>* d_out);

}  // namespace og
