// td_rng.cuh -- CPython-compatible MT19937 consumer for the scripted opponents (random.Random semantics:
// getrandbits, _randbelow, shuffle, random), drawing from the record's tempered word cache.
#pragma once
#include "td_common.cuh"

namespace td {

// ------------------------------------------------------------------------------------------------
// CPython-compatible MT19937 consumer (random.Random): one tempered window of <= 32 words per fill

// Regenerate the 624 words in place.  mt[k] = mt[(k+397)%624] ^ f(mt[k], mt[k+1]); chunks of 32 words in
// ascending order keep every operand in the state (old / new) the sequential algorithm sees.
__device__ __noinline__ void mt_twist(uint32_t *mt, int lane)
{
#pragma unroll 1
    for (int base = 0; base < kMtWords; base += kLanes) {
        const int k = base + lane;
        uint32_t v = 0;
        if (k < kMtWords - 1) {
            uint32_t y = (mt[k] & 0x80000000u) | (mt[k + 1] & 0x7fffffffu);
            v = mt[k < 227 ? k + 397 : k - 227] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
        }
        __syncwarp();
        if (k < kMtWords - 1) mt[k] = v;
        __syncwarp();
    }
    if (lane == 0) {
        uint32_t y = (mt[623] & 0x80000000u) | (mt[0] & 0x7fffffffu);
        mt[623] = mt[396] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
    }
    __syncwarp();
}

// The same through shared memory: the 20 dependent chunks of the regeneration cost one HBM round trip each when
// run on the state in place (40 us per twist under load); staged, the state travels once in and once out.
// gmt is 16-byte aligned (624 words per env), smt is a 2496-byte staging area in the warp's slice.
__device__ __noinline__ void mt_twist_staged(uint32_t *gmt, uint32_t *smt, int lane)
{
    for (int q = lane; q < kMtWords / 4; q += kLanes) reinterpret_cast<int4 *>(smt)[q] = reinterpret_cast<const int4 *>(gmt)[q];
    __syncwarp();
    mt_twist(smt, lane);
    for (int q = lane; q < kMtWords / 4; q += kLanes) reinterpret_cast<int4 *>(gmt)[q] = reinterpret_cast<const int4 *>(smt)[q];
    __syncwarp();
}

__device__ __forceinline__ uint32_t mt_temper(uint32_t y)
{
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
}

// The generator words of a step are consumed from the record's word cache, which holds TEMPERED words: a draw is
// one broadcast read from shared memory.  The cache is topped up behind the observation stores only when less
// than half of it is left (refill / finish_refill: most steps neither read the generator state nor write the cache
// back).  Only when a step needs more words than the cache holds (the scripted defender's shuffle, a few percent
// of its steps) the out-of-line refill fetches them from the generator state in HBM, twisting it when exhausted.
struct MtRefill { int cn, mt_pos; };
__device__ __noinline__ MtRefill mt_refill(uint32_t *cache, uint32_t *mt, uint32_t *stage, int lane, int mt_pos, int words)
{
    if (mt_pos >= kMtWords) { mt_twist_staged(mt, stage, lane); mt_pos = 0; }
    const int n = min(words, kMtWords - mt_pos);
    __syncwarp();                                       // every earlier read of the cache is done
    for (int q = lane; q < n; q += kLanes) cache[q] = mt_temper(mt[mt_pos + q]);
    __syncwarp();
    MtRefill r;
    r.cn = n;
    r.mt_pos = mt_pos;
    return r;
}

template <class W>
__device__ __forceinline__ void mt_more_words(W &w)
{
    const MtRefill r = mt_refill(const_cast<uint32_t *>(w.rng_cache()), w.mt, w.twist_stage(), w.lane, w.mt_pos,
                                 w.rng_words());
    w.cn = r.cn;
    w.mt_pos = r.mt_pos;
    w.ck = 0;
    w.cache_dirty = true;
}

// raw words just copied from the generator state -> tempered, in place
template <class W>
__device__ __forceinline__ void temper_cache(W &w)
{
    uint32_t *cache = const_cast<uint32_t *>(w.rng_cache());
    constexpr int kIters = W::kRngWords > 0 ? (W::kRngWords + kLanes - 1) / kLanes : 0;
    if (kIters > 0) {
#pragma unroll
        for (int it = 0; it < kIters; ++it) {
            const int q = w.lane + kLanes * it;
            if (q < w.cn) cache[q] = mt_temper(cache[q]);
        }
    } else {
        for (int q = w.lane; q < w.cn; q += kLanes) cache[q] = mt_temper(cache[q]);
    }
    __syncwarp();
}

template <class W>
__device__ __forceinline__ uint32_t mt_next(W &w)
{
    if (__builtin_expect(w.ck >= w.cn, 0)) mt_more_words(w);
    TD_CHECK(w, w.ck >= 0 && w.ck < w.cn && w.cn <= w.rng_words() && w.mt_pos < kMtWords);
    const uint32_t r = w.rng_cache()[w.ck];
    ++w.ck;
    ++w.mt_pos;
    return r;
}

// random._randbelow_with_getrandbits(n), 1 <= n < 2^31
template <class W>
__device__ __forceinline__ int py_randbelow(W &w, int n)
{
    const int shift = __clz(n);      // 32 - bit_length(n)
    uint32_t r;
    do { r = mt_next(w) >> shift; } while (r >= (uint32_t)n);
    return (int)r;
}

// random.shuffle(list) (for i in reversed(range(1, n)): j = randbelow(i + 1); swap) on a uint16 list in shared
// memory.  The draws are serial by definition (rejections shift every later draw), so one lane runs the whole
// loop alone, straight over the tempered word cache -- a fifth of the instructions of the same loop with a
// warp-wide draw per element.
template <class W>
__device__ __forceinline__ void py_shuffle_u16(W &w, uint16_t *list, int n)
{
    int i = n - 1;
    while (i >= 1) {
        if (w.ck >= w.cn) mt_more_words(w);
        TD_CHECK(w, w.cn <= w.rng_words() && w.mt_pos + (w.cn - w.ck) <= kMtWords);
        int k = w.ck;
        if (w.lane == 0) {
            const uint32_t *words = w.rng_cache();
            const int end = w.cn;
            while (i >= 1 && k < end) {
                const uint32_t r = words[k++] >> __clz(i + 1);
                if (r <= (uint32_t)i) {
                    const uint16_t t = list[i];
                    list[i] = list[r];
                    list[r] = t;
                    --i;
                }
            }
        }
        k = __shfl_sync(kFull, k, 0);
        i = __shfl_sync(kFull, i, 0);
        w.mt_pos += k - w.ck;
        w.ck = k;
        __syncwarp();
    }
}

template <class W>
__device__ __forceinline__ double py_random(W &w)
{
    uint32_t a = mt_next(w) >> 5, b = mt_next(w) >> 6;
    return __dmul_rn(__dadd_rn(__dmul_rn((double)a, 67108864.0), (double)b), 1.0 / 9007199254740992.0);
}

} // namespace td
