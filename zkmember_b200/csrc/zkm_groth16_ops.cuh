// zkm_groth16_ops.cuh -- what zkm_api.cu needs of the Groth16 proof assembly (zkm_groth16.cuh): the kernel arguments
// and the per-curve launchers.
#pragma once
#include "zkm_common.cuh"

namespace zkm {
// Groth16 proof assembly (zkm_groth16.cuh).  Key records (2 W + 1 words, flag word 1 = infinity): key1 = alpha_g1,
// beta_g1, delta_g1, a_query[0], b_g1_query[0]; key2 = beta_g2, delta_g2, b_g2_query[0].  rec[] = the five MSM records.
enum { G16_ALPHA = 0, G16_BETA, G16_DELTA, G16_A0, G16_B0 };
enum { G16_BETA2 = 0, G16_DELTA2, G16_B2_0 };
enum { G16_H = 0, G16_L, G16_A, G16_B1, G16_B2 };
struct G16Args {
    const uint64_t* key1;
    const uint64_t* key2;
    const uint64_t* rec[5];
    int rec_words[5];
    const uint32_t* range_flag;   // non-zero: an assignment element is not below the scalar modulus
    uint32_t r[12], s[12];        // the blinding scalars, canonical, 32-bit limbs
    uint64_t* out;                // A | B | C records, packed
};
struct G16Ops {
    size_t (*table_bytes)(int group);
    // window table of a finite delta (host record) into d_table
    void (*table)(Context* c, int group, const uint64_t* base_xy, char* d_table, cudaStream_t s);
    // *d_flag |= 1 if one of the n canonical scalars is >= r
    void (*range)(Context* c, const uint64_t* d_scalars, size_t n, uint32_t* d_flag, cudaStream_t s);
    // group 1: A and C (needs the four G1 records); group 2: B (needs all five); d_table: null when delta is the identity
    void (*assemble)(Context* c, int group, const G16Args& a, const char* d_table, cudaStream_t s);
};
G16Ops groth16_ops(int curve);

}  // namespace zkm
