// Packed coordinate keys and the atomics the search tables claim them with, shared by the A* table (pg_search.cu) and the
// level tables of the layered search (pg_layered.cu).  Coordinate i occupies key_bits bits at offset i * key_bits; a key of
// at most 63 bits is one word (KEYW = 1), of at most 127 bits two (KEYW = 2).
#pragma once
#include <stdint.h>

namespace {

template <int KEYW>
struct Key;
template <>
struct Key<1> {
    unsigned long long lo;
    __device__ __forceinline__ static Key zero() { return Key{0ull}; }
    __device__ __forceinline__ void add_bit(int off) { lo += 1ull << off; }
    __device__ __forceinline__ void add_val(unsigned v, int off) { lo += (unsigned long long)v << off; }
    __device__ __forceinline__ Key plus(const Key &o) const { return Key{lo + o.lo}; }
    __device__ __forceinline__ unsigned field(int off, unsigned m) const { return (unsigned)(lo >> off) & m; }
    // 32-bit multiplicative mix of the two key halves (the directory has at most 2^28 lines); the caller takes the TOP
    // bits, which every key bit reaches: two multiplies, one xor-shift, one more multiply
    __device__ __forceinline__ unsigned long long hash() const
    {
        unsigned h = (unsigned)lo * 0x9E3779B1u + (unsigned)(lo >> 32) * 0x85EBCA77u;
        h ^= h >> 15;
        h *= 0xC2B2AE3Du;
        return h;
    }
};
template <>
struct Key<2> {
    unsigned long long lo, hi;
    __device__ __forceinline__ static Key zero() { return Key{0ull, 0ull}; }
    __device__ __forceinline__ void add_val(unsigned v, int off)
    {
        unsigned __int128 x = ((unsigned __int128)hi << 64) | lo;
        x += (unsigned __int128)v << off;
        lo = (unsigned long long)x;
        hi = (unsigned long long)(x >> 64);
    }
    __device__ __forceinline__ void add_bit(int off) { add_val(1u, off); }
    __device__ __forceinline__ Key plus(const Key &o) const
    {
        unsigned __int128 x = (((unsigned __int128)hi << 64) | lo) + (((unsigned __int128)o.hi << 64) | o.lo);
        return Key{(unsigned long long)x, (unsigned long long)(x >> 64)};
    }
    __device__ __forceinline__ unsigned field(int off, unsigned m) const
    {
        unsigned __int128 x = ((unsigned __int128)hi << 64) | lo;
        return (unsigned)(x >> off) & m;
    }
    __device__ __forceinline__ unsigned long long hash() const
    {
        unsigned h = (unsigned)lo * 0x9E3779B1u + (unsigned)(lo >> 32) * 0x85EBCA77u + (unsigned)hi * 0x165667B1u +
                     (unsigned)(hi >> 32) * 0xD3A2646Cu;
        h ^= h >> 15;
        h *= 0xC2B2AE3Du;
        return h;
    }
};

__device__ __forceinline__ unsigned long long ld_cg_u64(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.global.cg.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void ld_cg_v2(const unsigned long long *p, unsigned long long &a, unsigned long long &b)
{
    asm volatile("ld.global.cg.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ void cas128(unsigned long long *addr, unsigned long long n0, unsigned long long n1, unsigned long long &o0,
                                       unsigned long long &o1)
{ // compare with {0,0}
    asm volatile(
        "{\n\t.reg .b128 c, n, o;\n\tmov.b128 c, {%3, %4};\n\tmov.b128 n, {%5, %6};\n\t"
        "atom.global.cas.b128 o, [%2], c, n;\n\tmov.b128 {%0, %1}, o;\n\t}"
        : "=l"(o0), "=l"(o1)
        : "l"(addr), "l"(0ull), "l"(0ull), "l"(n0), "l"(n1)
        : "memory");
}

} // namespace
