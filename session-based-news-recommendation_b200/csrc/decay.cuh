// Freshness decay of top-K recommendation (DESIGN §4.10): the one definition that the scoring GEMM's epilogue
// (score_fwd_pair_kernel<3>) and the exact re-scoring (recommend_scan_kernel<*, true>) share; util.decay_penalty is
// its host mirror.  Session b has a request time t_ref (int32, the clock unit of the item times) and a rate
// lambda >= 0 (finite fp32, score units per clock unit):
//   age(n) = min(max(t_ref - t[n], 0), TCAR_DECAY_MAX_AGE)     an exact integer, exact in fp32
//   p      = lambda * age                                      one fp32 multiply, round to nearest
//   r      = s - p                                             one fp32 subtract, round to nearest
// Items published after t_ref get age 0.  Ages saturate at TCAR_DECAY_MAX_AGE = 2^23 - 1 clock units (about 16 years
// in minutes): that bound makes the conversion exact whatever the int32 inputs, and lets it run without I2F (the XU
// pipe) -- the float with the bits 0x4B000000 + a is 2^23 + a for 0 <= a < 2^23, so age = that float - 2^23 with
// the row-constant bits = 0x4B000000 + t_ref: two IMNMX, one IADD and one FADD per score.
// __fmul_rn / __fsub_rn keep the compiler from contracting the multiply and the subtract into one FFMA.
#pragma once
#include <stdint.h>
#include "tcar_b200.h"

namespace tcar {

struct DecayRow {
    int32_t ref;      // t_ref
    int32_t lo;       // the latest time whose age saturates: max(t_ref - TCAR_DECAY_MAX_AGE, INT32_MIN)
    uint32_t bits;    // 0x4B000000 + t_ref (mod 2^32)
    float rate;       // lambda
};

__device__ __forceinline__ DecayRow decay_row(int32_t t_ref, float rate) {
    DecayRow d;
    d.ref = t_ref;
    d.lo = t_ref < INT32_MIN + TCAR_DECAY_MAX_AGE ? INT32_MIN : t_ref - TCAR_DECAY_MAX_AGE;
    d.bits = 0x4B000000u + (uint32_t)t_ref;
    d.rate = rate;
    return d;
}

// age(n) as fp32: t_ref - clamp(t, lo, t_ref) lies in [0, 2^23), so the integer subtract of the clamped time from
// `bits` is 0x4B000000 + age
__device__ __forceinline__ float decay_age(const DecayRow& d, int32_t t) {
    const int32_t c = max(min(t, d.ref), d.lo);
    return __fsub_rn(__uint_as_float(d.bits - (uint32_t)c), 8388608.f);
}

// r = s - lambda * age
__device__ __forceinline__ float decayed(float s, const DecayRow& d, int32_t t) {
    return __fsub_rn(s, __fmul_rn(d.rate, decay_age(d, t)));
}

}  // namespace tcar
