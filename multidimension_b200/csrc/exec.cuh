// exec.cuh — per-thread evaluator of a lowered View chain (device code).
//
// One thread computes V consecutive output elements along the innermost output axis ("a
// vector").  The op tree is a postfix program over a small value stack held in REGISTERS:
// every function here is force-inlined into a context where the stack depth D is a compile-time
// constant, so `st[D][lane]` never needs dynamic indexing.  Two drivers use it:
//   * run_static<Sig,...>  — the instruction stream (opcode,dtype,op,aux) is a compile-time
//     signature; the compiler folds every switch away.  This is the device-side analogue of the
//     reference's monomorphisation of `Zip<Map<..>>` types into one `collect` loop.
//   * run_interp<...>      — `switch (depth)` into the same code with run-time opcodes, for any
//     chain without a pre-instantiated signature.
//
// When compiled without __CUDACC__ (tests/emu only) the same source runs on the host, one
// "thread" at a time, so planner + evaluator logic can be checked against the oracle on a box
// without a GPU.  That build is test infrastructure and is never linked into the product.
#pragma once
#include <stdint.h>
#include <string.h>

#include "program.hpp"

#if defined(__CUDACC__)
#define MDIM_FN __device__ __forceinline__
#define MDIM_CE __host__ __device__ constexpr
#else
#include <math.h>
#define MDIM_FN static inline __attribute__((always_inline))
#define MDIM_CE constexpr
#endif

// SHAPE-LIKE fields of the program (ranks, lengths, strides, dividers, predicate forms, opcodes' slot
// numbers) are read through MDIM_SHAPE_OF(P).  Normally that is the run-time program itself; the run-time
// specialiser (jit.cu) can instead point it at a `constexpr Program` generated for one concrete shape, which
// turns every stride into an immediate, drops zero strides and length-1 axes, and makes every divider a
// compile-time constant.  Pointers, offsets and immediates always come from the real program.
#ifndef MDIM_SHAPE_OF
#define MDIM_SHAPE_OF(P) (P)
#endif

namespace mdim {

// ------------------------------------------------------------------------------------------------
// scalar helpers
// ------------------------------------------------------------------------------------------------
MDIM_FN float as_f32(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
MDIM_FN uint32_t f32_bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
MDIM_FN double as_f64(uint64_t u) { double f; memcpy(&f, &u, 8); return f; }
MDIM_FN uint64_t f64_bits(double f) { uint64_t u; memcpy(&u, &f, 8); return u; }

// Rust never contracts `x*y+1.0` into an FMA and rounds every operation separately
// (SURVEY.md §7 hard part 7): use the explicit round-to-nearest intrinsics, which nvcc never fuses.
#if defined(__CUDA_ARCH__)
MDIM_FN float f_add(float a, float b) { return __fadd_rn(a, b); }
MDIM_FN float f_sub(float a, float b) { return __fsub_rn(a, b); }
MDIM_FN float f_mul(float a, float b) { return __fmul_rn(a, b); }
MDIM_FN float f_div(float a, float b) { return __fdiv_rn(a, b); }
MDIM_FN double d_add(double a, double b) { return __dadd_rn(a, b); }
MDIM_FN double d_sub(double a, double b) { return __dsub_rn(a, b); }
MDIM_FN double d_mul(double a, double b) { return __dmul_rn(a, b); }
MDIM_FN double d_div(double a, double b) { return __ddiv_rn(a, b); }
#else
MDIM_FN float f_add(float a, float b) { volatile float r = a + b; return r; }
MDIM_FN float f_sub(float a, float b) { volatile float r = a - b; return r; }
MDIM_FN float f_mul(float a, float b) { volatile float r = a * b; return r; }
MDIM_FN float f_div(float a, float b) { volatile float r = a / b; return r; }
MDIM_FN double d_add(double a, double b) { volatile double r = a + b; return r; }
MDIM_FN double d_sub(double a, double b) { volatile double r = a - b; return r; }
MDIM_FN double d_mul(double a, double b) { volatile double r = a * b; return r; }
MDIM_FN double d_div(double a, double b) { volatile double r = a / b; return r; }
#endif

MDIM_FN int esize_of(int dt) { return dt == MDIM_U8 ? 1 : (dt == MDIM_I32 || dt == MDIM_U32 || dt == MDIM_F32) ? 4 : 8; }

// ------------------------------------------------------------------------------------------------
// global memory access.  Streaming vector loads bypass L1 (read once); scalar broadcast / strided /
// gather loads go through L1 (re-used across lanes and neighbouring threads).
// ------------------------------------------------------------------------------------------------
#if defined(__CUDA_ARCH__)
MDIM_FN void ld128_stream(const void* p, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "l"(p));
}
MDIM_FN void ld128_cached(const void* p, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
    asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "l"(p));
}
// 256-bit accesses (new on sm_100): one instruction moves a thread's whole 32-byte vector, so a warp
// instruction covers 1 KB of whole sectors.  With two 128-bit accesses per thread every instruction touches
// HALF of each 32-byte sector: harmless for reads, but a write-only stream then runs at 4.0 instead of
// 7.6 TB/s (profiles/: iota collect), and the write-bound rank-5 chain at 4.2 instead of 6.4.
#if defined(MDIM_NO_VEC256)  // an NVRTC older than 12.9 (PTX < 8.8) has no 256-bit vector accesses: two 128-bit ones
MDIM_FN void ld256_stream(const void* p, uint32_t (&r)[8]) { ld128_stream(p, r[0], r[1], r[2], r[3]); ld128_stream((const char*)p + 16, r[4], r[5], r[6], r[7]); }
MDIM_FN void ld256_cached(const void* p, uint32_t (&r)[8]) { ld128_cached(p, r[0], r[1], r[2], r[3]); ld128_cached((const char*)p + 16, r[4], r[5], r[6], r[7]); }
#else
MDIM_FN void ld256_stream(const void* p, uint32_t (&r)[8]) {
    asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "l"(p));
}
MDIM_FN void ld256_cached(const void* p, uint32_t (&r)[8]) {
    asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "l"(p));
}
#endif
#if defined(MDIM_NO_VEC256)
MDIM_FN void st128(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d, bool cs);
MDIM_FN void st256(void* p, const uint32_t (&r)[8], bool cs) { st128(p, r[0], r[1], r[2], r[3], cs); st128((char*)p + 16, r[4], r[5], r[6], r[7], cs); }
#else
MDIM_FN void st256(void* p, const uint32_t (&r)[8], bool cs) {
    if (cs) asm volatile("st.global.cs.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
    else asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
#endif
MDIM_FN void ld64_stream(const void* p, uint32_t& a, uint32_t& b) {
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(a), "=r"(b) : "l"(p));
}
MDIM_FN uint32_t ld32_stream(const void* p) {
    uint32_t a; asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(a) : "l"(p)); return a;
}
MDIM_FN uint32_t ld32(const void* p) { return __ldg((const uint32_t*)p); }
MDIM_FN uint64_t ld64(const void* p) { return __ldg((const unsigned long long*)p); }
// Random reads of a source far larger than L2: ask L2 for 64 bytes per miss instead of the whole 128-byte line.
// Measured (profiles/r2_gather_probe.md, 2^28 uniform-random 4-byte reads over 4 GiB): DRAM reads 72 instead of 134 bytes
// per element, 5.66 instead of 6.04 ms.  Slower than the plain load when the source (partly) fits in L2, hence the flag.
MDIM_FN uint32_t ld32_big(const void* p) { uint32_t a; asm volatile("ld.global.nc.L2::64B.u32 %0, [%1];" : "=r"(a) : "l"(p)); return a; }
MDIM_FN uint64_t ld64_big(const void* p) { unsigned long long a; asm volatile("ld.global.nc.L2::64B.u64 %0, [%1];" : "=l"(a) : "l"(p)); return a; }
MDIM_FN uint32_t ld8(const void* p) { return __ldg((const uint8_t*)p); }
MDIM_FN void st128(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d, bool cs) {
    if (cs) asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
    else asm volatile("st.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
MDIM_FN void st64(void* p, uint32_t a, uint32_t b) {
    asm volatile("st.global.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(a), "r"(b) : "memory");
}
MDIM_FN void st32(void* p, uint32_t a) { *(uint32_t*)p = a; }
MDIM_FN void st8(void* p, uint32_t a) { *(uint8_t*)p = (uint8_t)a; }
MDIM_FN void err_min(unsigned long long* p, unsigned long long v) { atomicMin(p, v); }
#else
MDIM_FN void ld128_stream(const void* p, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
    const uint32_t* q = (const uint32_t*)p; a = q[0]; b = q[1]; c = q[2]; d = q[3];
}
MDIM_FN void ld128_cached(const void* p, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) { ld128_stream(p, a, b, c, d); }
MDIM_FN void ld256_stream(const void* p, uint32_t (&r)[8]) { memcpy(r, p, 32); }
MDIM_FN void ld256_cached(const void* p, uint32_t (&r)[8]) { memcpy(r, p, 32); }
MDIM_FN void st256(void* p, const uint32_t (&r)[8], bool) { memcpy(p, r, 32); }
MDIM_FN void ld64_stream(const void* p, uint32_t& a, uint32_t& b) { const uint32_t* q = (const uint32_t*)p; a = q[0]; b = q[1]; }
MDIM_FN uint32_t ld32_stream(const void* p) { return *(const uint32_t*)p; }
MDIM_FN uint32_t ld32(const void* p) { return *(const uint32_t*)p; }
MDIM_FN uint64_t ld64(const void* p) { return *(const uint64_t*)p; }
MDIM_FN uint32_t ld32_big(const void* p) { return *(const uint32_t*)p; }
MDIM_FN uint64_t ld64_big(const void* p) { return *(const uint64_t*)p; }
MDIM_FN uint32_t ld8(const void* p) { return *(const uint8_t*)p; }
MDIM_FN void st128(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d, bool) { uint32_t* q = (uint32_t*)p; q[0] = a; q[1] = b; q[2] = c; q[3] = d; }
MDIM_FN void st64(void* p, uint32_t a, uint32_t b) { uint32_t* q = (uint32_t*)p; q[0] = a; q[1] = b; }
MDIM_FN void st32(void* p, uint32_t a) { *(uint32_t*)p = a; }
MDIM_FN void st8(void* p, uint32_t a) { *(uint8_t*)p = (uint8_t)a; }
MDIM_FN void err_min(unsigned long long* p, unsigned long long v) { if (v < *p) *p = v; }
#endif

template <bool CACHED> MDIM_FN void ld128(const void* p, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
    if constexpr (CACHED) ld128_cached(p, a, b, c, d); else ld128_stream(p, a, b, c, d);
}

template <class S> MDIM_FN S ld_scalar_big(const void* base, int64_t idx, int esize) {
    if (esize == 4) return (S)ld32_big((const char*)base + idx * 4);
    if (esize == 1) return (S)ld8((const char*)base + idx);
    if (sizeof(S) == 8) return (S)ld64_big((const char*)base + idx * 8);
    return 0;
}

template <class S> MDIM_FN S ld_scalar(const void* base, int64_t idx, int esize) {
    if (esize == 4) return (S)ld32((const char*)base + idx * 4);
    if (esize == 1) return (S)ld8((const char*)base + idx);
    if (sizeof(S) == 8) return (S)ld64((const char*)base + idx * 8);
    return 0;
}

// V consecutive elements starting at element `idx`; the planner guarantees the alignment.
template <class S, int V, bool CACHED> MDIM_FN void ld_vector(const void* base, int64_t idx, int esize, S (&d)[V], bool w256 = false) {
    if constexpr (V * sizeof(S) == 32 && (sizeof(S) == 4 || sizeof(S) == 8)) {
        if (w256 && esize == (int)sizeof(S)) {  // the whole 32-byte vector in one access
            uint32_t r[8];
            if constexpr (CACHED) ld256_cached((const char*)base + idx * esize, r); else ld256_stream((const char*)base + idx * esize, r);
            if constexpr (sizeof(S) == 4) {
#pragma unroll
                for (int i = 0; i < 8; ++i) d[i] = (S)r[i];
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) d[i] = (S)r[2 * i] | ((S)r[2 * i + 1] << 32);
            }
            return;
        }
    }
    if (esize == 4) {
        const char* p = (const char*)base + idx * 4;
        if constexpr (V % 4 == 0) {
#pragma unroll
            for (int i = 0; i < V; i += 4) {
                uint32_t a, b, c, e;
                ld128<CACHED>(p + i * 4, a, b, c, e);
                d[i] = a; d[i + 1] = b; d[i + 2] = c; d[i + 3] = e;
            }
        } else if constexpr (V == 2) {
            uint32_t a, b; ld64_stream(p, a, b); d[0] = a; d[1] = b;
        } else {
            d[0] = ld32_stream(p);
        }
    } else if (esize == 8) {
        if constexpr (sizeof(S) == 8) {
            const char* p = (const char*)base + idx * 8;
            if constexpr (V % 2 == 0) {
#pragma unroll
                for (int i = 0; i < V; i += 2) {
                    uint32_t a, b, c, e;
                    ld128<CACHED>(p + i * 8, a, b, c, e);
                    d[i] = (S)a | ((S)b << 32); d[i + 1] = (S)c | ((S)e << 32);
                }
            } else {
                uint32_t a, b; ld64_stream(p, a, b); d[0] = (S)a | ((S)b << 32);
            }
        }
    } else {
        const char* p = (const char*)base + idx;
        if constexpr (V == 8) {
            uint32_t a, b; ld64_stream(p, a, b);
#pragma unroll
            for (int i = 0; i < 4; ++i) { d[i] = (a >> (8 * i)) & 0xffu; d[4 + i] = (b >> (8 * i)) & 0xffu; }
        } else if constexpr (V == 4) {
            uint32_t a = ld32_stream(p);
#pragma unroll
            for (int i = 0; i < 4; ++i) d[i] = (a >> (8 * i)) & 0xffu;
        } else {
#pragma unroll
            for (int i = 0; i < V; ++i) d[i] = (S)ld8(p + i);
        }
    }
}

// Wide stores are streaming (st.global.cs, evict-first): nothing re-reads the output.
template <class S, int V> MDIM_FN void st_vector(void* base, uint64_t idx, int esize, const S (&d)[V], bool w256 = false) {
    if constexpr (V * sizeof(S) == 32 && (sizeof(S) == 4 || sizeof(S) == 8)) {
        if (w256 && esize == (int)sizeof(S)) {
            uint32_t r[8];
            if constexpr (sizeof(S) == 4) {
#pragma unroll
                for (int i = 0; i < 8; ++i) r[i] = (uint32_t)d[i];
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) { r[2 * i] = (uint32_t)d[i]; r[2 * i + 1] = (uint32_t)((uint64_t)d[i] >> 32); }
            }
            st256((char*)base + idx * esize, r, true);
            return;
        }
    }
    if (esize == 4) {
        char* p = (char*)base + idx * 4;
        if constexpr (V % 4 == 0) {
#pragma unroll
            for (int i = 0; i < V; i += 4) st128(p + i * 4, (uint32_t)d[i], (uint32_t)d[i + 1], (uint32_t)d[i + 2], (uint32_t)d[i + 3], true);
        } else if constexpr (V == 2) {
            st64(p, (uint32_t)d[0], (uint32_t)d[1]);
        } else {
            st32(p, (uint32_t)d[0]);
        }
    } else if (esize == 8) {
        if constexpr (sizeof(S) == 8) {
            char* p = (char*)base + idx * 8;
            if constexpr (V % 2 == 0) {
#pragma unroll
                for (int i = 0; i < V; i += 2)
                    st128(p + i * 8, (uint32_t)d[i], (uint32_t)(d[i] >> 32), (uint32_t)d[i + 1], (uint32_t)(d[i + 1] >> 32), true);
            } else {
                st64(p, (uint32_t)d[0], (uint32_t)(d[0] >> 32));
            }
        }
    } else {
        char* p = (char*)base + idx;
        if constexpr (V == 8) {
            uint32_t a = 0, b = 0;
#pragma unroll
            for (int i = 0; i < 4; ++i) { a |= ((uint32_t)d[i] & 0xffu) << (8 * i); b |= ((uint32_t)d[4 + i] & 0xffu) << (8 * i); }
            st64(p, a, b);
        } else if constexpr (V == 4) {
            uint32_t a = 0;
#pragma unroll
            for (int i = 0; i < 4; ++i) a |= ((uint32_t)d[i] & 0xffu) << (8 * i);
            st32(p, a);
        } else {
#pragma unroll
            for (int i = 0; i < V; ++i) st8(p + i, (uint32_t)d[i]);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// value semantics.  A slot holds the raw bits of one value, zero-extended to the slot width.
// Integer semantics follow Rust RELEASE builds: add/sub/mul wrap, shift amounts are masked,
// x/0 and MIN/-1 panic in every build mode (→ arith error).  Floats are IEEE, never fused.
// ------------------------------------------------------------------------------------------------
template <class S> MDIM_FN S bin_op(int dt, int op, int rdt, S a, S b, bool& arith) {
    if (dt == MDIM_F32) {
        float x = as_f32((uint32_t)a), y = as_f32((uint32_t)b), r = 0.f;
        switch (op) {
            case MDIM_ADD: r = f_add(x, y); break;
            case MDIM_SUB: r = f_sub(x, y); break;
            case MDIM_MUL: r = f_mul(x, y); break;
            case MDIM_DIV: r = f_div(x, y); break;
            case MDIM_REM: r = fmodf(x, y); break;  // Rust f32 % is fmod, exact
        }
        return (S)f32_bits(r);
    }
    if (dt == MDIM_I32 || dt == MDIM_U32 || dt == MDIM_U8) {
        uint32_t x = (uint32_t)a, y = (uint32_t)b, r = 0;
        const uint32_t bits = dt == MDIM_U8 ? 8u : 32u;
        switch (op) {
            case MDIM_ADD: r = x + y; break;
            case MDIM_SUB: r = x - y; break;
            case MDIM_MUL: r = x * y; break;
            case MDIM_AND: r = x & y; break;
            case MDIM_OR: r = x | y; break;
            case MDIM_XOR: r = x ^ y; break;
            case MDIM_SHL: r = x << ((uint32_t)b & (bits - 1)); break;  // low bits of any rhs dtype
            case MDIM_SHR:
                r = dt == MDIM_I32 ? (uint32_t)((int32_t)x >> ((uint32_t)b & 31u)) : x >> ((uint32_t)b & (bits - 1));
                break;
            case MDIM_DIV:
            case MDIM_REM:
                if (y == 0 || (dt == MDIM_I32 && x == 0x80000000u && y == 0xffffffffu)) { arith = true; r = 0; }
                else if (dt == MDIM_I32) r = op == MDIM_DIV ? (uint32_t)((int32_t)x / (int32_t)y) : (uint32_t)((int32_t)x % (int32_t)y);
                else r = op == MDIM_DIV ? x / y : x % y;
                break;
        }
        if (dt == MDIM_U8) r &= 0xffu;
        (void)rdt;
        return (S)r;
    }
    if constexpr (sizeof(S) == 8) {
        if (dt == MDIM_F64) {
            double x = as_f64(a), y = as_f64(b), r = 0.;
            switch (op) {
                case MDIM_ADD: r = d_add(x, y); break;
                case MDIM_SUB: r = d_sub(x, y); break;
                case MDIM_MUL: r = d_mul(x, y); break;
                case MDIM_DIV: r = d_div(x, y); break;
                case MDIM_REM: r = fmod(x, y); break;
            }
            return f64_bits(r);
        }
        uint64_t x = a, y = b, r = 0;
        switch (op) {
            case MDIM_ADD: r = x + y; break;
            case MDIM_SUB: r = x - y; break;
            case MDIM_MUL: r = x * y; break;
            case MDIM_AND: r = x & y; break;
            case MDIM_OR: r = x | y; break;
            case MDIM_XOR: r = x ^ y; break;
            case MDIM_SHL: r = x << (y & 63u); break;
            case MDIM_SHR: r = dt == MDIM_I64 ? (uint64_t)((int64_t)x >> (y & 63u)) : x >> (y & 63u); break;
            case MDIM_DIV:
            case MDIM_REM:
                if (y == 0 || (dt == MDIM_I64 && x == 0x8000000000000000ull && y == ~0ull)) { arith = true; r = 0; }
                else if (dt == MDIM_I64) r = op == MDIM_DIV ? (uint64_t)((int64_t)x / (int64_t)y) : (uint64_t)((int64_t)x % (int64_t)y);
                else r = op == MDIM_DIV ? x / y : x % y;
                break;
        }
        return r;
    }
    return 0;
}

// Rust `as`: float→int saturates and maps NaN to 0; int→int truncates / sign-extends;
// int→float rounds to nearest even.
MDIM_FN int64_t sat_i64(double f, int64_t lo, int64_t hi) {
    if (f != f) return 0;
    if (f <= (double)lo) return lo;
    if (f >= (double)hi) return hi;
    return (int64_t)f;
}
MDIM_FN uint64_t sat_u64(double f, uint64_t hi) {
    if (f != f || f <= 0.0) return 0;
    if (f >= (double)hi) return hi;
    return (uint64_t)f;
}

template <class S> MDIM_FN S cast_val(int from, int to, S a) {
    if (from == to) return a;
    const bool from_f = from == MDIM_F32 || from == MDIM_F64;
    if (from_f) {
        double d;
        if (from == MDIM_F32) d = (double)as_f32((uint32_t)a);
        else { if constexpr (sizeof(S) == 8) d = as_f64(a); else d = 0.; }
        switch (to) {
            case MDIM_U8: return (S)sat_u64(d, 255);
            case MDIM_I32: return (S)(uint32_t)(int32_t)sat_i64(d, INT32_MIN, INT32_MAX);
            case MDIM_U32: return (S)sat_u64(d, 0xffffffffull);
            case MDIM_I64: return (S)(uint64_t)sat_i64(d, INT64_MIN, INT64_MAX);
            case MDIM_U64: return (S)sat_u64(d, ~0ull);
            case MDIM_F32: return (S)f32_bits((float)d);
            case MDIM_F64: if constexpr (sizeof(S) == 8) return f64_bits(d); else return 0;
        }
        return 0;
    }
    // integer source: canonical 64-bit two's complement value
    uint64_t bits;
    bool sgn = false;
    switch (from) {
        case MDIM_I32: bits = (uint64_t)(int64_t)(int32_t)(uint32_t)a; sgn = true; break;
        case MDIM_I64: bits = (uint64_t)a; sgn = true; break;
        default: bits = (uint64_t)a; break;
    }
    switch (to) {
        case MDIM_U8: return (S)(bits & 0xffu);
        case MDIM_I32: case MDIM_U32: return (S)(uint32_t)bits;
        case MDIM_I64: case MDIM_U64: return (S)bits;
        case MDIM_F32: return (S)f32_bits(sgn ? (float)(int64_t)bits : (float)bits);
        case MDIM_F64: if constexpr (sizeof(S) == 8) return f64_bits(sgn ? (double)(int64_t)bits : (double)bits); else return 0;
    }
    return 0;
}

template <class S> MDIM_FN S un_op(int op, int dt, int src_dt, S a) {
    if (op == MDIM_CAST) return cast_val<S>(src_dt, dt, a);
    if (dt == MDIM_F32) {
        float x = as_f32((uint32_t)a);
        switch (op) {
            case MDIM_NEG: return (S)(f32_bits(x) ^ 0x80000000u);
            case MDIM_ABS: return (S)(f32_bits(x) & 0x7fffffffu);
            case MDIM_SQRT: return (S)f32_bits(sqrtf(x));
        }
        return a;
    }
    if (dt == MDIM_F64) {
        if constexpr (sizeof(S) == 8) {
            switch (op) {
                case MDIM_NEG: return a ^ 0x8000000000000000ull;
                case MDIM_ABS: return a & 0x7fffffffffffffffull;
                case MDIM_SQRT: return f64_bits(sqrt(as_f64(a)));
            }
        }
        return a;
    }
    if (dt == MDIM_I64 || dt == MDIM_U64) {
        if constexpr (sizeof(S) == 8) {
            switch (op) {
                case MDIM_NEG: return (S)(0ull - a);
                case MDIM_NOT: return (S)~a;
                case MDIM_ABS: return (dt == MDIM_I64 && (int64_t)a < 0) ? (S)(0ull - a) : a;
            }
        }
        return a;
    }
    uint32_t x = (uint32_t)a, r = x;
    switch (op) {
        case MDIM_NEG: r = 0u - x; break;
        case MDIM_NOT: r = ~x; break;
        case MDIM_ABS: r = (dt == MDIM_I32 && (int32_t)x < 0) ? 0u - x : x; break;
    }
    if (dt == MDIM_U8) r &= 0xffu;
    return (S)r;
}

// ------------------------------------------------------------------------------------------------
// per-thread state.  MAXR = number of iteration axes this instantiation walks (the planner picks the
// smallest instantiation >= rank + red_rank; axes beyond the program's own have length 1, stride 0,
// so no loop below ever tests the run-time rank).  MAXR == 1 is the contiguous stream form.
// WIDE = 64-bit coordinates and offsets; otherwise the planner has proved that every coordinate,
// every per-operand linear offset and every predicate value fits in 32 bits.
// ------------------------------------------------------------------------------------------------
template <bool WIDE> struct CoordTraits { using coord_t = uint32_t; using off_t = int32_t; };
template <> struct CoordTraits<true> { using coord_t = uint64_t; using off_t = int64_t; };

template <bool WIDE, int MAXR> struct ThreadState {
    typename CoordTraits<WIDE>::coord_t c[MAXR];  // element coordinates of lane 0
    typename CoordTraits<WIDE>::coord_t rk;       // coordinate along the fastest reduction axis
    uint64_t pos0;                                // linear output position of lane 0
    uint64_t red_k;                               // reduction step counter
    uint32_t mask;                                // lane-active mask (Diagonal laziness)
};

// offset + sum_a coord[a] * stride[a]: Index::to_usize of the operand's own index (src/index.rs:109-114)
// after every Transpose/Iso/Row/Column/broadcast remapping has been folded into the strides.
template <bool WIDE, int MAXR>
MDIM_FN typename CoordTraits<WIDE>::off_t addr_offset(const Program& P, int slot, const ThreadState<WIDE, MAXR>& ts) {
    using off_t = typename CoordTraits<WIDE>::off_t;
    off_t off = (off_t)P.addr[slot].offset + (off_t)ts.rk * (off_t)MDIM_SHAPE_OF(P).addr[slot].rstride;
#pragma unroll
    for (int a = 0; a < MAXR; ++a) off += (off_t)ts.c[a] * (off_t)MDIM_SHAPE_OF(P).addr[slot].stride[a];
    return off;
}

MDIM_FN int64_t inner_stride(const Program& P, int slot) { (void)P; return MDIM_SHAPE_OF(P).addr[slot].inner; }

// Predicates are linear forms: sum_a coef[a] * coord[a] (+ lane * lane_coef) == rhs.
// `coord[a] == coord[b]` is coef[a] = 1, coef[b] = -1, rhs = 0; `coord[a] == k` is coef[a] = 1, rhs = k.
template <int V, bool WIDE, int MAXR>
MDIM_FN uint32_t eval_preds(const Program& P, const ThreadState<WIDE, MAXR>& ts, int first, int n) {
    using off_t = typename CoordTraits<WIDE>::off_t;
    uint32_t m = (1u << V) - 1u;
    for (int p = first; p < first + n; ++p) {
        off_t s = (off_t)ts.rk * (off_t)MDIM_SHAPE_OF(P).pred[p].rcoef;
#pragma unroll
        for (int a = 0; a < MAXR; ++a) s += (off_t)ts.c[a] * (off_t)MDIM_SHAPE_OF(P).pred[p].coef[a];
        const off_t rhs = (off_t)MDIM_SHAPE_OF(P).pred[p].rhs, lc = (off_t)MDIM_SHAPE_OF(P).pred[p].lane_coef;
        // cmp 0: ==   1: <   2: >=   — evaluated with plain integer logic: a (uniform) branch per predicate
        // here keeps the compiler from hoisting the operand loads that follow, which cost config 5 17 %.
        const uint32_t is_eq = (uint32_t)(MDIM_SHAPE_OF(P).pred[p].cmp == 0), want_neg = (uint32_t)(MDIM_SHAPE_OF(P).pred[p].cmp == 1);
        if (lc == 0) {  // the vector axis is not involved: one test for all lanes
            const off_t d = s - rhs;
            const uint32_t zero = (uint32_t)(d == 0), neg = (uint32_t)(d < 0);
            const uint32_t ok = (is_eq & zero) | ((1u ^ is_eq) & (1u ^ neg ^ want_neg));
            m &= 0u - ok;
        } else {
#pragma unroll
            for (int l = 0; l < V; ++l) {
                const off_t d = s + (off_t)l * lc - rhs;
                const uint32_t zero = (uint32_t)(d == 0), neg = (uint32_t)(d < 0);
                const uint32_t ok = (is_eq & zero) | ((1u ^ is_eq) & (1u ^ neg ^ want_neg));
                m &= ~((1u ^ ok) << l);
            }
        }
    }
    return m;
}

MDIM_FN void report(const Program& P, ErrWord* err, uint64_t pos, int status, int node, int comp, uint64_t value, uint64_t bound) {
    err_min(&err->pos, (unsigned long long)pos);
    if ((P.flags & PF_EXPLAIN) && pos == P.explain_pos && err->status == 0) {
        err->status = status; err->node = node; err->component = comp;
        err->value = value; err->bound = bound;
    }
}

// depth change of one instruction
MDIM_FN int depth_delta(int opc, int aux) {
    switch (opc) {
        case OPC_FOLD_BEGIN: return aux == 1 ? 0 : 1;  // aux 1: the initial value is already on the stack (FOLD with an init view)
        case OPC_LEAF_VEC: case OPC_LEAF_BCAST: case OPC_LEAF_STRIDED: case OPC_IOTA: case OPC_CONST: return 1;
        case OPC_BINARY: case OPC_FOLD_STEP: case OPC_SELECT2: return -1;
        case OPC_GATHER: return 1 - aux;
        default: return 0;
    }
}

// GATHER with NC index components at st[D-NC .. D-1]; result replaces st[D-NC].
// Compose::at = w.at(v.at(i)) (src/view.rs:905,911); each component is bounds-checked like
// usize::to_usize (src/int.rs:16-19) in component order; inactive (off-diagonal) lanes neither
// load nor report, because Diagonal::at never evaluates its inner view there (src/view.rs:854-856).
template <int D, int NC, class S, int V, int MAXD, bool WIDE, int MAXR>
MDIM_FN void exec_gather(const Program& P, ErrWord* err, const Instr& I, int slot, S (&st)[MAXD][V], const ThreadState<WIDE, MAXR>& ts) {
    if constexpr (sizeof(S) == 8 && D >= NC && NC >= 1) {
        const Addr& A = MDIM_SHAPE_OF(P).addr[slot];  // gstride / bound / n_peers: shape-like; the pointer is read from P
        const int64_t base = (int64_t)addr_offset<WIDE, MAXR>(P, slot, ts);
        const int64_t s_in = inner_stride(P, slot);
        const int es = esize_of(I.dtype);
#pragma unroll
        for (int l = 0; l < V; ++l) {
            int64_t idx = base + (int64_t)l * s_in;
            bool ok = (ts.mask >> l) & 1u;
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                const uint64_t k = (uint64_t)st[D - NC + c][l];
                if (ok && !(k < A.bound[c])) {
                    report(P, err, ts.pos0 + l, MDIM_ERR_OOB, I.n, c, k, A.bound[c]);
                    ok = false;
                }
                idx += (int64_t)k * A.gstride[c];
            }
            S v = 0;
            if (ok) {
                if (A.n_peers > 1) {
                    const uint64_t p = (uint64_t)idx / P.peers.block;
                    v = ld_scalar<S>(P.peers.peer[p], (int64_t)((uint64_t)idx - p * P.peers.block), es);
                } else if (P.flags & PF_GATHER_BIG) {
                    v = ld_scalar_big<S>(P.addr[slot].ptr, idx, es);
                } else {
                    v = ld_scalar<S>(P.addr[slot].ptr, idx, es);
                }
            }
            st[D - NC][l] = v;
        }
    }
}

// One step of Index::each over the reduction axes, last axis fastest (src/index.rs:122-124): the fastest
// axis is the counter rk; only when it wraps do the slower axes (kept in c[]) move.
template <bool WIDE, int MAXR> MDIM_FN void carry_red(const Program& P, ThreadState<WIDE, MAXR>& ts) {
    bool carry = true;
#pragma unroll
    for (int a = MAXR - 1; a >= 0; --a) {
        if (carry && a >= MDIM_SHAPE_OF(P).rank && a < MDIM_SHAPE_OF(P).rank + MDIM_SHAPE_OF(P).red_rank) {
            ts.c[a] += 1;
            if ((uint64_t)ts.c[a] >= MDIM_SHAPE_OF(P).length[a]) ts.c[a] = 0; else carry = false;
        }
    }
}
template <bool WIDE, int MAXR> MDIM_FN void advance_red(const Program& P, ThreadState<WIDE, MAXR>& ts) {
    ts.rk += 1;
    if ((uint64_t)ts.rk >= MDIM_SHAPE_OF(P).red_fast_len) { ts.rk = 0; carry_red<WIDE, MAXR>(P, ts); }
}

// Execute instruction I at compile-time stack depth D.  Returns the next pc.
// SLOTK >= 0: the address slot is known at compile time (static signatures: slots are handed out in
// instruction order, so it is the number of addressed instructions before this one).  Reading it from the
// program instead makes every stride a register-indexed constant load (LDC) rather than a uniform one.
// A LEAF whose Array is sharded over the GPUs of the box (instruction aux bit 1; mdim_node.n_peers): element `off`
// of the whole Array lives at peers.peer[off / block] + off % block.  Vectors never straddle two blocks (the
// planner only vectorises when block boundaries are vector-aligned).
template <bool WIDE> MDIM_FN const void* leaf_base(const Program& P, int slot, int aux, int64_t& off) {
    if (aux & 2) {
        uint64_t p;
        if constexpr (WIDE) p = (uint64_t)off / P.peers.block;
        else p = (uint32_t)off / (uint32_t)P.peers.block;  // 32-bit coordinates: every offset is below 2^31
        off -= (int64_t)(p * P.peers.block);
        return P.peers.peer[p];
    }
    return P.addr[slot].ptr;
}

template <int D, class S, int V, int MAXD, bool WIDE, int MAXR, int SLOTK = -1>
MDIM_FN int exec_instr(const Program& P, ErrWord* err, int opc, int dtype, int op, int aux, int pc,
                       S (&st)[MAXD][V], ThreadState<WIDE, MAXR>& ts) {
    const Instr& I = MDIM_SHAPE_OF(P).instr[pc];  // opcode operands (slot, n, source node) are shape-like ...
    const uint64_t imm = P.instr[pc].imm;          // ... immediates are run-time data
    const int slot = SLOTK >= 0 ? SLOTK : (int)I.slot;  // (address slot; MASK / SELECT read I.slot themselves)
    int next = pc + 1;
    switch (opc) {
        case OPC_LEAF_VEC:  // Array::at = items[to_usize(index)] (src/array.rs:81,86), V at a time
            if constexpr (D < MAXD) {
                int64_t off = (int64_t)addr_offset<WIDE, MAXR>(P, slot, ts);
                const void* base = leaf_base<WIDE>(P, slot, aux, off);
                if (ts.mask == (1u << V) - 1u) {  // (a compile-time fact in signatures without MASK)
                    const bool w256 = (P.flags & PF_VEC256) != 0;
                    if (aux & 1) ld_vector<S, V, true>(base, off, esize_of(dtype), st[D], w256);   // re-read operand: keep in L1
                    else ld_vector<S, V, false>(base, off, esize_of(dtype), st[D], w256);          // read once: stream past L1
                } else {  // under a Concat / lazy Diagonal: inactive lanes must not touch memory
                    const int es = esize_of(dtype);
#pragma unroll
                    for (int l = 0; l < V; ++l) st[D][l] = ((ts.mask >> l) & 1u) ? ld_scalar<S>(base, off + l, es) : (S)0;
                }
            }
            break;
        case OPC_LEAF_BCAST:  // operand lacks the vector axis: Broadcast::index drops it (src/broadcast.rs:46-60)
            if constexpr (D < MAXD) {
                int64_t off = (int64_t)addr_offset<WIDE, MAXR>(P, slot, ts);
                const void* base = leaf_base<WIDE>(P, slot, aux, off);
                const S v = ts.mask ? ld_scalar<S>(base, off, esize_of(dtype)) : (S)0;
#pragma unroll
                for (int l = 0; l < V; ++l) st[D][l] = v;
            }
            break;
        case OPC_LEAF_STRIDED:
            if constexpr (D < MAXD) {
                const int64_t off = (int64_t)addr_offset<WIDE, MAXR>(P, slot, ts), s_in = inner_stride(P, slot);
                const int es = esize_of(dtype);
#pragma unroll
                for (int l = 0; l < V; ++l) {
                    int64_t o = off + (int64_t)l * s_in;  // (a sharded operand: the lanes may belong to different peers)
                    const void* base = leaf_base<WIDE>(P, slot, aux, o);
                    st[D][l] = ((ts.mask >> l) & 1u) ? ld_scalar<S>(base, o, es) : (S)0;
                }
            }
            break;
        case OPC_IOTA:  // All<I>::at(index) = index (src/index.rs:185)
            if constexpr (D < MAXD) {
                const int64_t off = (int64_t)addr_offset<WIDE, MAXR>(P, slot, ts), s_in = inner_stride(P, slot);
#pragma unroll
                for (int l = 0; l < V; ++l) {
                    const uint64_t x = (uint64_t)(off + (int64_t)l * s_in);
                    if constexpr (sizeof(S) == 8) st[D][l] = cast_val<S>(MDIM_U64, dtype, x);
                    else st[D][l] = dtype == MDIM_F32 ? (S)f32_bits((float)x) : dtype == MDIM_U8 ? (S)(x & 0xffu) : (S)(uint32_t)x;
                }
            }
            break;
        case OPC_CONST:  // Scalar::at (src/view.rs:1407)
            if constexpr (D < MAXD) {
#pragma unroll
                for (int l = 0; l < V; ++l) st[D][l] = (S)imm;
            }
            break;
        case OPC_UNARY:  // Map::at = f(v.at(i)) (src/view.rs:888), closed op set
            if constexpr (D >= 1) {
#pragma unroll
                for (int l = 0; l < V; ++l) st[D - 1][l] = un_op<S>(op, dtype, aux, st[D - 1][l]);
            }
            break;
        case OPC_BINARY:  // Zip::at = B::call(v.at(vi), w.at(wi)) (src/view.rs:1194-1197)
            if constexpr (D >= 2) {
#pragma unroll
                for (int l = 0; l < V; ++l) {
                    bool arith = false;
                    st[D - 2][l] = bin_op<S>(dtype, op, aux, st[D - 2][l], st[D - 1][l], arith);
                    if (arith && ((ts.mask >> l) & 1u)) report(P, err, ts.pos0 + l, MDIM_ERR_ARITH, I.n, 0, (uint64_t)st[D - 1][l], 0);
                }
            }
            break;
        case OPC_MASK:
            ts.mask = I.n ? eval_preds<V, WIDE, MAXR>(P, ts, I.slot, I.n) : ((1u << V) - 1u);
            break;
        case OPC_SELECT:  // Diagonal::at (src/view.rs:854-856)
            if constexpr (D >= 1) {
                const uint32_t m = eval_preds<V, WIDE, MAXR>(P, ts, I.slot, I.n);
#pragma unroll
                for (int l = 0; l < V; ++l) st[D - 1][l] = ((m >> l) & 1u) ? st[D - 1][l] : (S)imm;
            }
            break;
        case OPC_SELECT2:  // Concat::at (src/view.rs:938-945): V where coord < len(V), else W
            if constexpr (D >= 2) {
                const uint32_t m = eval_preds<V, WIDE, MAXR>(P, ts, I.slot, 1);
#pragma unroll
                for (int l = 0; l < V; ++l) st[D - 2][l] = ((m >> l) & 1u) ? st[D - 2][l] : st[D - 1][l];
            }
            break;
        case OPC_GATHER:
            if (aux == 1) exec_gather<D, 1, S, V, MAXD, WIDE, MAXR>(P, err, I, slot, st, ts);
            else if (aux == 2) exec_gather<D, 2, S, V, MAXD, WIDE, MAXR>(P, err, I, slot, st, ts);
            else if (aux == 3) exec_gather<D, 3, S, V, MAXD, WIDE, MAXR>(P, err, I, slot, st, ts);
            break;
        case OPC_FOLD_BEGIN:  // let mut s = init;  (the closure of rows().map(..), SURVEY.md fact 3)
            if constexpr (D < MAXD) {
                if (aux != 1) {
#pragma unroll
                    for (int l = 0; l < V; ++l) st[D][l] = (S)imm;
                }
#pragma unroll
                for (int a = 0; a < MAXR; ++a)
                    if (a >= MDIM_SHAPE_OF(P).rank) ts.c[a] = 0;
                ts.red_k = 0;
                ts.rk = 0;
                if (MDIM_SHAPE_OF(P).red_count == 0) next = I.slot;  // empty row: skip the body and its FOLD_STEP
            }
            break;
        case OPC_FOLD_STEP:  // row.each(|x| s = s (op) x): sequential, index order (src/view.rs:250-252)
            if constexpr (D >= 2) {
#pragma unroll
                for (int l = 0; l < V; ++l) {
                    bool arith = false;
                    st[D - 2][l] = bin_op<S>(dtype, op, aux, st[D - 2][l], st[D - 1][l], arith);
                    if (arith && ((ts.mask >> l) & 1u)) report(P, err, ts.pos0 + l, MDIM_ERR_ARITH, I.n, 0, (uint64_t)st[D - 1][l], 0);
                }
                advance_red<WIDE, MAXR>(P, ts);
                ts.red_k += 1;
                if (ts.red_k < MDIM_SHAPE_OF(P).red_count) next = I.slot;
            }
            break;
    }
    return next;
}

// ------------------------------------------------------------------------------------------------
// drivers
// ------------------------------------------------------------------------------------------------
// compile-time signature: Sig::n instructions, Sig::code[i] = {opc, dtype, op, aux}
struct SigInstr { uint8_t opc, dtype, op, aux; };

struct NoSig { static constexpr int n = 0; };

// index of the FOLD_STEP that closes the FOLD_BEGIN at `pc` (folds do not nest)
template <class Sig> MDIM_CE int sig_fold_end(int pc) {
    for (int i = pc + 1; i < Sig::n; ++i)
        if (Sig::code[i].opc == OPC_FOLD_STEP) return i;
    return Sig::n;
}
MDIM_CE bool sig_is_addressed(SigInstr I) {
    return I.opc == OPC_LEAF_VEC || I.opc == OPC_LEAF_BCAST || I.opc == OPC_LEAF_STRIDED || I.opc == OPC_IOTA || I.opc == OPC_GATHER;
}
// address slot of instruction `pc`: plan.cpp hands slots out in instruction order
template <class Sig> MDIM_CE int sig_addr_slot(int pc) {
    int k = 0;
    for (int i = 0; i < pc; ++i)
        if (sig_is_addressed(Sig::code[i])) ++k;
    return sig_is_addressed(Sig::code[pc]) ? k : -1;
}
MDIM_CE int sig_depth_after(SigInstr I, int d) {
    return d + (I.opc == OPC_LEAF_VEC || I.opc == OPC_LEAF_BCAST || I.opc == OPC_LEAF_STRIDED || I.opc == OPC_IOTA || I.opc == OPC_CONST ||
                        (I.opc == OPC_FOLD_BEGIN && I.aux != 1) ? 1
                : I.opc == OPC_BINARY || I.opc == OPC_FOLD_STEP || I.opc == OPC_SELECT2 ? -1
                : I.opc == OPC_GATHER ? 1 - (int)I.aux
                                      : 0);
}

// Runs instructions [PC, STOP) of the signature at compile-time depth D.  A fold becomes a real loop:
//   FOLD_BEGIN; for k in 0..red_count { body; FOLD_STEP }   — sequential, index order (src/view.rs:250-252)
template <class Sig, int PC, int D, int STOP, class S, int V, int MAXD, bool WIDE, int MAXR>
MDIM_FN void run_static(const Program& P, ErrWord* err, S (&st)[MAXD][V], ThreadState<WIDE, MAXR>& ts) {
    if constexpr (PC < STOP) {
        constexpr SigInstr I = Sig::code[PC];
        if constexpr (I.opc == OPC_FOLD_BEGIN) {
            constexpr int END = sig_fold_end<Sig>(PC);
            constexpr int B = I.aux == 1 ? D - 1 : D;  // stack slot of the accumulator (aux 1: the init view's value, already pushed)
            exec_instr<D, S, V, MAXD, WIDE, MAXR>(P, err, I.opc, I.dtype, I.op, I.aux, PC, st, ts);
            constexpr SigInstr E = Sig::code[END < Sig::n ? END : PC];
            // Outer loop: the slower reduction axes (coordinates in c[], rare).  Inner loop: the fastest one,
            // where every coordinate in c[] is loop-invariant, so an operand's address is base + rk * rstride;
            // unrolled so that several steps' loads (independent of the add chain) are in flight together.
            const uint64_t outer = MDIM_SHAPE_OF(P).red_fast_len ? MDIM_SHAPE_OF(P).red_count / MDIM_SHAPE_OF(P).red_fast_len : 0;
            for (uint64_t ko = 0; ko < outer; ++ko) {
#pragma unroll 8
                for (uint64_t k = 0; k < MDIM_SHAPE_OF(P).red_fast_len; ++k) {
                    ts.rk = (typename CoordTraits<WIDE>::coord_t)k;
                    run_static<Sig, PC + 1, B + 1, END, S, V, MAXD, WIDE, MAXR>(P, err, st, ts);
                    if constexpr (B >= 0 && B + 2 <= MAXD) {
#pragma unroll
                        for (int l = 0; l < V; ++l) {
                            bool arith = false;
                            st[B][l] = bin_op<S>(E.dtype, E.op, E.aux, st[B][l], st[B + 1][l], arith);
                            if (arith && ((ts.mask >> l) & 1u)) report(P, err, ts.pos0 + l, MDIM_ERR_ARITH, P.instr[END].n, 0, (uint64_t)st[B + 1][l], 0);
                        }
                    }
                }
                ts.rk = 0;
                carry_red<WIDE, MAXR>(P, ts);
            }
            run_static<Sig, END + 1, B + 1, STOP, S, V, MAXD, WIDE, MAXR>(P, err, st, ts);
        } else {
            exec_instr<D, S, V, MAXD, WIDE, MAXR, sig_addr_slot<Sig>(PC)>(P, err, I.opc, I.dtype, I.op, I.aux, PC, st, ts);
            run_static<Sig, PC + 1, sig_depth_after(I, D), STOP, S, V, MAXD, WIDE, MAXR>(P, err, st, ts);
        }
    }
}

template <int D, class S, int V, int MAXD, bool WIDE, int MAXR>
MDIM_FN int interp_step(const Program& P, ErrWord* err, int depth, const Instr& I, int pc, S (&st)[MAXD][V], ThreadState<WIDE, MAXR>& ts) {
    if constexpr (D > MAXD) {
        return P.n_instr;  // unreachable: the planner bounds the depth
    } else {
        if (depth == D) return exec_instr<D, S, V, MAXD, WIDE, MAXR>(P, err, I.opc, I.dtype, I.op, I.aux, pc, st, ts);
        return interp_step<D + 1, S, V, MAXD, WIDE, MAXR>(P, err, depth, I, pc, st, ts);
    }
}

template <class S, int V, int MAXD, bool WIDE, int MAXR>
MDIM_FN void run_interp(const Program& P, ErrWord* err, S (&st)[MAXD][V], ThreadState<WIDE, MAXR>& ts) {
    int pc = 0, depth = 0;
    while (pc < P.n_instr) {
        const Instr& I = P.instr[pc];
        const int d = depth_delta(I.opc, I.aux);
        pc = interp_step<0, S, V, MAXD, WIDE, MAXR>(P, err, depth, I, pc, st, ts);
        depth += d;
    }
}

// Fast unsigned division by a run-time constant for n < 2^31 (planner guarantees the range):
// q = umulhi(n, mul) >> shr.  mul == 0 encodes division by 1.
MDIM_FN uint32_t fast_div(uint32_t n, uint32_t mul, uint32_t shr) {
#if defined(__CUDA_ARCH__)
    return mul ? __umulhi(n, mul) >> shr : n;
#else
    return mul ? (uint32_t)(((uint64_t)n * mul) >> 32) >> shr : n;
#endif
}

// One output vector: decode (Index::from_usize peels the LAST component first, src/index.rs:116-120,
// src/lib.rs:38-39), evaluate, store at its to_usize position (row-major, src/index.rs:109-114).
// Program axis 0 is the vector axis, so the decode runs a = 0, 1, ...: dec_len[a] is the decode length
// of axis a (axis 0 counted in vectors of V elements; 1 for reduction / unused axes) and
// dec_scale[a] turns the decoded count back into an element coordinate.
template <class Sig, class S, int V, int MAXD, bool WIDE, int MAXR>
MDIM_FN void eval_vector(const Program& P, void* out, ErrWord* err, uint64_t g) {
    using coord_t = typename CoordTraits<WIDE>::coord_t;
    ThreadState<WIDE, MAXR> ts;
    ts.pos0 = g * (uint64_t)V;
    ts.mask = (1u << V) - 1u;
    ts.red_k = 0;
    ts.rk = 0;
    coord_t rem = (coord_t)g;
#pragma unroll
    for (int a = 0; a < MAXR - 1; ++a) {  // axis 0 = the vector axis, peeled first
        coord_t q;
        if constexpr (WIDE) q = rem / (coord_t)MDIM_SHAPE_OF(P).dec_len[a];
        else q = fast_div(rem, MDIM_SHAPE_OF(P).div_mul[a], MDIM_SHAPE_OF(P).div_shr[a]);
        const coord_t r = rem - q * (coord_t)MDIM_SHAPE_OF(P).dec_len[a];
        ts.c[a] = r * (coord_t)MDIM_SHAPE_OF(P).dec_scale[a];
        rem = q;
    }
    ts.c[MAXR - 1] = rem * (coord_t)MDIM_SHAPE_OF(P).dec_scale[MAXR - 1];
    S st[MAXD][V];
    if constexpr (Sig::n > 0) run_static<Sig, 0, 0, Sig::n, S, V, MAXD, WIDE, MAXR>(P, err, st, ts);
    else run_interp<S, V, MAXD, WIDE, MAXR>(P, err, st, ts);
    st_vector<S, V>(out, ts.pos0, esize_of(MDIM_SHAPE_OF(P).out_dtype), st[0], (P.flags & PF_VEC256) != 0);
    if (MDIM_SHAPE_OF(P).n_out > 1) {  // a tuple-typed root: value k of the final stack is scalar leaf k, stored to its own run
#pragma unroll
        for (int k = 1; k < MDIM_MAX_OUTS; ++k)
            if (k < MAXD && k < MDIM_SHAPE_OF(P).n_out)
                st_vector<S, V>(P.out_more[k - 1], ts.pos0, esize_of(MDIM_SHAPE_OF(P).out_dtypes[k]), st[k < MAXD ? k : 0]);
    }
}

}  // namespace mdim
