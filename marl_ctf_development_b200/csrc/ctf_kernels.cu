// ctf_kernels.cu — sm_100a kernels and C ABI of the batched GridworldCtf step path.
//
// One warp owns one environment.  The env's tile map is staged in shared memory
// (16-byte-row layout, 256 B), agent i lives in the registers of lane i, and the
// reference's sequential semantics (gridworld_ctf.py:849-918) are kept by
// iterating the dice-ordered agents serially while using the lanes for the
// parallel inner parts: per-opponent tag tests (ballot), the 3x3 respawn window
// (ballot + nth-set-bit), proximity metrics (ballot + popc), state staging and
// the observation writer.  Observations (standardise_state, :975-1009) are built
// as one bit per output element in shared memory — only non-open cells set bits —
// and streamed to HBM with 128-bit stores, so the kernel's cost is the store
// stream, not the logic.
//
// Randomness is Philox4x32-10 addressed by (seed, global env id, episode, step,
// site); see marl_ctf_development_b200/draws.py for the site map.  Lane l of the
// warp generates site l.
#include <cuda.h>           // driver API types of the compressible allocator (entry points come through the runtime)
#include <cudaTypedefs.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>   // snprintf for error messages
#include <string.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <new>
#include <type_traits>
#include <unordered_map>

#include "../../include/ctf_b200.h"

// Resident CTAs per SM of k_step when it writes observation deltas (ctf_bind_obs_record; see ctf_create).  Set on the
// nvcc command line only to build the libraries of a residency sweep (tools/obs_delta_bench.py --cap-lib).
#ifndef CTF_DELTA_CTAS_PER_SM
#define CTF_DELTA_CTAS_PER_SM 9
#endif

namespace {

constexpr int kWarpsPerCta = 4;   // 2 warps per CTA tie with 4, 8 and 16 lose (see k_step)
constexpr int kThreads = kWarpsPerCta * 32;
constexpr int kRow = 16;       // shared/global grid row stride (cells)
constexpr int kGridBytes = 256;
constexpr int kMaxList = 256;  // non-open cell list entries
constexpr unsigned kFull = 0xFFFFFFFFu;

// Everything the kernels need, derived from ctf_config_t on the host in ctf_create().
struct DevPlan {
    unsigned long long tag_threshold;
    unsigned long long lut64[2];  // 4 bits per tile code -> channel, per observer team
    double reward_step, reward_capture, reward_tag, capture_punish, win_margin, loss_margin;
    int G, N, C, GG, M, E;        // E = N*C*G*G observation elements per env
    int bits_words;               // words of the per-env observation bit string (alignment pad + slack, multiple of 16)
    int wpa;                      // words per agent of the packed observation output: ceil(C*G*G / 32)
    int game_steps, flip_axis;
    int flip_a, flip_b, flip_d;    // flipped cell index = flip_a * r + flip_b * c + flip_d
    int use_adjusted_rewards, home_flag_capture, drop_flag_when_no_hp, reverse_team1_actions;
    int heal_q, vault_cost_q, vault_min_q;
    int zone_distance, guardian_distance, tagging_range, max_agent_blocks, block_pickup_value;
    int hp_max_q[4], damage_q[4], damage_boosted_q[4];
    // hp_float: HP as IEEE doubles, every operation rounded like the reference's Python floats (non-dyadic configs)
    int hp_float;
    double hp_max_f[4], damage_f[4], damage_boosted_f[4], heal_f, vault_cost_f, vault_min_f;
    int warp_smem_bytes, list_off, bits_off;
    unsigned char team[8], type[8], tile[8], start_r[8], start_c[8], obs_rev[8], meta_hp_src[8];
    signed char my_slot[8];        // index of agent i in OPPONENTS[1 - team(i)], -1 if truncated away
    unsigned char n_opp[2];
    unsigned char flag_pos[2][2], capture_pos[2][2], spawn_pos[2][2], flag_tile[2];
    signed char delta[4][9][2];
    unsigned char rev_action[16];
    unsigned int meta_row[8];        // metadata slots of observer a: nibble q -> agent id (0xF = none)
    unsigned int meta_codes[64];     // kMeta* code of every element of the [N][M] metadata block, four per word
    unsigned char grid_template[kGridBytes];  // 16-stride rows
};

struct Launch {
    // state
    uint8_t* grid;
    unsigned long long* agents;
    uint4* envs;
    uint32_t* stats;
    uint8_t* visits;
    double* hp;             // [B][N] when plan.hp_float
    // outputs
    void* obs;
    uint32_t* obs_bits;
    float* meta;
    float* rewards;
    uint8_t* dones;
    const uint8_t* actions;
    uint32_t* faults;
    // record of `obs` (ctf_bind_obs_record; all null unless outputs.obs is the bound buffer): the padded bit string
    // each env's last launch wrote into obs ([B][bits_words]), the epoch it was written in ([B]) and the current epoch
    uint32_t* record;
    uint32_t* record_epoch;
    const uint32_t* epoch;
    long long B;
    uint32_t seed_lo, seed_hi;
    uint32_t env_id_base;
    uint32_t rev_override;  // bit 8 set: bits 0..7 replace plan.obs_rev
    int first_reset;
};

// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t (&out)[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__device__ __forceinline__ int cheb(int r0, int c0, int r1, int c1) { return max(abs(r0 - r1), abs(c0 - c1)); }

// lane-register form of one agent: row | col<<4 | has_flag<<8 | hp_q<<16 (int16)
__device__ __forceinline__ uint32_t pack_agent(int r, int c, int flag, int hp) {
    return (uint32_t)r | ((uint32_t)c << 4) | ((uint32_t)flag << 8) | ((uint32_t)(hp & 0xFFFF) << 16);
}
__device__ __forceinline__ int ag_r(uint32_t m) { return m & 15; }
__device__ __forceinline__ int ag_c(uint32_t m) { return (m >> 4) & 15; }
__device__ __forceinline__ int ag_flag(uint32_t m) { return (m >> 8) & 1; }
__device__ __forceinline__ int ag_hp(uint32_t m) { return (int)(short)(m >> 16); }

struct WarpMem {
    uint8_t* grid;     // [256]
    uint32_t* list;    // [256]
    uint32_t* bits;    // [bits_words]
};

__device__ __forceinline__ WarpMem warp_mem(const DevPlan& P, unsigned char* smem, int warp) {
    unsigned char* base = smem + (size_t)warp * P.warp_smem_bytes;
    WarpMem w;
    w.grid = base;
    w.list = reinterpret_cast<uint32_t*>(base + P.list_off);
    w.bits = reinterpret_cast<uint32_t*>(base + P.bits_off);
    return w;
}

// flipped destination cell of (r, c) for a reversed view (gridworld_ctf.py:1003-1007); all four maps are involutions
// and affine in (r, c): the host folds FLIP_AXIS into three coefficients (build_plan)
__device__ __forceinline__ int flip_cell(const DevPlan& P, int r, int c) { return P.flip_a * r + P.flip_b * c + P.flip_d; }

// ------------------------------------------------------------------------------------------------
// Observation + metadata writer (standardise_state :975-1009, get_env_metadata :1027-1069)
// ------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ uint4 expand_bits(uint32_t b);

template <>
__device__ __forceinline__ uint4 expand_bits<float>(uint32_t b) {  // 4 elements
    uint4 v;
    // 1.0f = 0x3F800000 has 23 trailing zero bits, so (b & 2^k) * (0x3F800000 >> k) is exact for k <= 3
    v.x = (b & 1u) * 0x3F800000u;
    v.y = (b & 2u) * 0x1FC00000u;
    v.z = (b & 4u) * 0x0FE00000u;
    v.w = (b & 8u) * 0x07F00000u;
    return v;
}

// 8 elements of a 16-bit float type whose 1.0 is ONE: word k packs bits 2k (low half) and 2k+1 (high half)
template <uint32_t ONE>
__device__ __forceinline__ uint4 expand_bits16(uint32_t b) {
    uint4 v;
    v.x = (((b & 3u) * 0x8001u) & 0x10001u) * ONE;
    v.y = ((((b >> 2) & 3u) * 0x8001u) & 0x10001u) * ONE;
    v.z = ((((b >> 4) & 3u) * 0x8001u) & 0x10001u) * ONE;
    v.w = ((((b >> 6) & 3u) * 0x8001u) & 0x10001u) * ONE;
    return v;
}
template <>
__device__ __forceinline__ uint4 expand_bits<__half>(uint32_t b) { return expand_bits16<0x3C00u>(b); }
template <>
__device__ __forceinline__ uint4 expand_bits<__nv_bfloat16>(uint32_t b) { return expand_bits16<0x3F80u>(b); }

template <typename T>
__device__ __forceinline__ T from_bit(uint32_t bit) { return (T)bit; }
template <>
__device__ __forceinline__ __half from_bit<__half>(uint32_t bit) { return __ushort_as_half((unsigned short)(bit ? 0x3C00u : 0u)); }
template <>
__device__ __forceinline__ __nv_bfloat16 from_bit<__nv_bfloat16>(uint32_t bit) {
    return __ushort_as_bfloat16((unsigned short)(bit ? 0x3F80u : 0u));
}

// Builds the env's observation block as one bit per element in shared memory (w.bits): element
// e = (a*C + c)*G*G + p of the [N][C][G][G] block is bit e.
// `pad` (obs_pad of the output block) shifts the whole string: element e is bit pad + e, so that the store vectors,
// counted from the alignment boundary below the block, cover whole nibbles / bytes / half-words of the string.
__device__ __forceinline__ void build_obs_bits(const DevPlan& P, const WarpMem& w, uint32_t me, uint32_t rev_mask, int pad, int lane) {
    const int N = P.N, GG = P.GG, CGG = P.C * P.GG;
    // 1. clear the bit string
    {
        uint4* b4 = reinterpret_cast<uint4*>(w.bits);
        const int n4 = (P.bits_words + 3) >> 2;
        for (int i = lane; i < n4; i += 32) b4[i] = make_uint4(0, 0, 0, 0);
    }
    // 2. list the non-open cells: channel(team-0 view) | channel(team-1 view)<<4 | dest(normal)<<8 | dest(flipped)<<16
    int count = 0;
#pragma unroll
    for (int j = 0; j < kGridBytes / 32; ++j) {
        const int cell = j * 32 + lane;
        const uint32_t t = w.grid[cell];
        const unsigned nz = __ballot_sync(kFull, t != 0);
        if (t != 0) {
            const int r = cell >> 4, c = cell & 15;
            const int pos = count + __popc(nz & ((1u << lane) - 1u));
            const uint32_t ch0 = (uint32_t)(P.lut64[0] >> (t * 4)) & 15u, ch1 = (uint32_t)(P.lut64[1] >> (t * 4)) & 15u;
            w.list[pos] = ch0 | (ch1 << 4) | ((uint32_t)(r * P.G + c) << 8) | ((uint32_t)flip_cell(P, r, c) << 16);
        }
        count += __popc(nz);
    }
    __syncwarp();
    // 3. scatter: lane l works for agent (l & 7) on list entries (l >> 3), (l >> 3) + 4, ...; lane a < N also sets
    //    agent a's own position plane (channel 0) from its registers
    {
        const int a = lane & 7;
        const bool valid = a < N;
        const bool rev = (rev_mask >> a) & 1u;
        const int ch_shift = P.team[a] ? 4 : 0, p_shift = rev ? 16 : 8;
        const int base = pad + a * CGG;
        for (int k = lane >> 3; k < count; k += 4) {
            const uint32_t ent = w.list[k];
            const int ch = (ent >> ch_shift) & 15;
            if (valid && ch) {
                const int e = base + ch * GG + (int)((ent >> p_shift) & 0xFFu);
                atomicOr(&w.bits[e >> 5], 1u << (e & 31));
            }
        }
        if (lane < N) {
            const int r = ag_r(me), c = ag_c(me);
            const int e = base + (rev ? flip_cell(P, r, c) : r * P.G + c);
            atomicOr(&w.bits[e >> 5], 1u << (e & 31));
        }
    }
    __syncwarp();
}

// One 128-bit vector of the observation stream.  A plain write-back store: 4 % faster than .cs for this stream (L2 merges
// and schedules the write-backs; profiles/r01_ab_store_op.log); evict-first hints are 5-8 % slower (r02_ab_l2_hints.log).
__device__ __forceinline__ void store_vec(uint4* p, uint4 v) { *p = v; }

// elements (= bits of the string) per 128-bit store
template <typename T>
constexpr int kVecElems = 16 / (int)sizeof(T);

// Alignment unit of the store vectors: a 32-byte sector.  Measured on one B200 (profiles/r02_ab_pad.log, ms per step
// 8_arena B=65536 / 7_gridlocked B=65536 / B=16384): 16 B -> 1.003 / 0.618 / 0.173, 32 B -> 1.003 / 0.551 / 0.151,
// 128 B -> 1.035 / 0.569 / 0.154: whole sectors matter (a sector shared by two store instructions is written twice
// into L2), whole lines do not.
constexpr int kPadBytes = 32;
// number of elements between the previous kPadBytes boundary and `out`: 0 .. kPadBytes / sizeof(T) - 1
template <typename T>
__device__ __forceinline__ int obs_pad(const T* out) {
    return (int)((reinterpret_cast<uintptr_t>(out) & (uintptr_t)(kPadBytes - 1)) / sizeof(T));
}

// uint8 stream: expand 8 bits -> 8 bytes with one 64-bit shared load from a 256-entry table.
// Bytes at the start of a kernel's dynamic shared memory taken by the expansion table of element type T.
template <typename T>
constexpr int kLutBytes = sizeof(T) == 1 ? 2048 : 0;

// Fills the table (all threads of the CTA, before any thread leaves the kernel); returns it, or nullptr for other types.
template <typename T>
__device__ __forceinline__ const uint2* init_expand_lut(uint4* smem_raw) {
    if constexpr (kLutBytes<T> > 0) {
        uint2* lut = reinterpret_cast<uint2*>(smem_raw);
        for (unsigned i = threadIdx.x; i < 256u; i += blockDim.x)
            lut[i] = make_uint2(((i & 15u) * 0x00204081u) & 0x01010101u, ((i >> 4) * 0x00204081u) & 0x01010101u);
        __syncthreads();
        return lut;
    } else {
        return nullptr;
    }
}

// Store vector v of a padded bit string (elements = bits VB*v .. VB*v + VB - 1).
template <typename T>
__device__ __forceinline__ uint4 vector_value(const uint32_t* __restrict__ bits, int v, const uint2* __restrict__ lut) {
    if constexpr (kLutBytes<T> > 0) {
        // uint8: the vector's 16 bits are two table lookups (8 bits -> 8 bytes each) instead of sixteen ALU operations
        const uint32_t h = bits[v >> 1] >> ((v & 1) * 16);
        const uint2 lo = lut[h & 0xFFu], hi = lut[(h >> 8) & 0xFFu];
        return make_uint4(lo.x, lo.y, hi.x, hi.y);
    } else {
        constexpr int VB = kVecElems<T>, VW = 32 / VB;
        return expand_bits<T>(bits[v / VW] >> ((v % VW) * VB));
    }
}

// The fewer than VB elements of a block before its first full vector and after its last one, as scalar stores
// (one warp).
template <typename T>
__device__ __forceinline__ void stream_edges(const uint32_t* __restrict__ bits, int nbits, T* __restrict__ out, int v_begin,
                                             int v_end, int lane) {
    constexpr int VB = kVecElems<T>;
    const int pad = obs_pad(out), total = pad + nbits;
    const int head_n = min(v_begin * VB - pad, nbits);          // < VB elements before the first full vector
    if (lane < head_n) out[lane] = from_bit<T>((bits[(pad + lane) >> 5] >> ((pad + lane) & 31)) & 1u);
    const int t = max(v_end * VB, pad + head_n) + lane;         // first bit covered by neither head nor full vectors
    if (t < total) out[t - pad] = from_bit<T>((bits[t >> 5] >> (t & 31)) & 1u);
}

// Stores the full vectors [v_begin, v_end) of a padded bit string (vector v = bits VB*v .. VB*v + VB - 1) at vp[v];
// warp `wi` of `nw` cooperating warps.  `bits` must be 16-byte aligned and readable up to a multiple of 16 words.
template <typename T>
__device__ __forceinline__ void stream_vectors(const uint32_t* __restrict__ bits, uint4* __restrict__ vp, int v_begin,
                                               int v_end, int wi, int nw, int lane, const uint2* __restrict__ lut) {
    if constexpr (sizeof(T) == 4) {
        // group g = 128 vectors = 16 words = 2 KB of output: lane (q, n) = (lane >> 3, lane & 7) reads words
        // 16g + 4q .. +3 with ONE 128-bit shared load and stores vector 8 * (16g + 4q + m) + n for m = 0..3, so every
        // store instruction writes four complete 128-byte runs.  The per-store bounds checks stay on purpose: a loop
        // without them (and with the next group's load issued early) executes 40 % fewer instructions but is 1 - 7 %
        // SLOWER (profiles/r02_ab_stream_loop*.log) — the HBM write stream likes stores spaced out, not bursts of four
        const int q = lane >> 3, n = lane & 7, sh = n * 4;
        const int n_groups = (v_end + 127) >> 7;
#pragma unroll 2
        for (int g = wi; g < n_groups; g += nw) {
            const uint4 wd = *reinterpret_cast<const uint4*>(bits + 16 * g + 4 * q);
            const int v0 = 128 * g + 32 * q + n;
            if (v0 >= v_begin && v0 < v_end) store_vec(vp + v0, expand_bits<T>(wd.x >> sh));
            if (v0 + 8 < v_end) store_vec(vp + v0 + 8, expand_bits<T>(wd.y >> sh));
            if (v0 + 16 < v_end) store_vec(vp + v0 + 16, expand_bits<T>(wd.z >> sh));
            if (v0 + 24 < v_end) store_vec(vp + v0 + 24, expand_bits<T>(wd.w >> sh));
        }
    } else {
#pragma unroll 4
        for (int v = wi * 32 + lane; v < v_end; v += nw * 32)
            if (v >= v_begin) store_vec(vp + v, vector_value<T>(bits, v, lut));
    }
}

// Streams `nbits` elements to `out` (any element alignment) from a bit string built with pad = obs_pad(out), i.e.
// laid out from the kPadBytes boundary below `out`: store vectors are then sector-aligned whatever the block's
// alignment (7_gridlocked's 52 728-byte env blocks start at every multiple of 8 bytes), no 32-byte sector is shared
// by two store instructions.  Vectors that lie completely inside the block go out as 128-bit stores, the
// fewer than VB elements before the first / after the last full vector as scalar stores (their neighbours belong
// to other envs).
template <typename T>
__device__ __forceinline__ void stream_env(const uint32_t* __restrict__ bits, int nbits, T* __restrict__ out, int wi, int nw,
                                           int lane, const uint2* __restrict__ lut) {
    constexpr int VB = kVecElems<T>;
    const int pad = obs_pad(out);
    const int total = pad + nbits;
    const int v_begin = (pad + VB - 1) / VB, v_end = total / VB;   // vectors counted from the alignment boundary
    if (wi == 0) stream_edges<T>(bits, nbits, out, v_begin, v_end, lane);
    stream_vectors<T>(bits, reinterpret_cast<uint4*>(out - pad), v_begin, v_end, wi, nw, lane, lut);
}

// Delta form of stream_env for a block whose previous bit string (same pad) is `rec`: only the 32-byte sectors whose
// bits differ from `rec` are stored, and only the 16-byte pieces of `rec` that differ are written back.  The string is
// taken in chunks of 128 words (a 16-byte piece per lane, 4 KB of float32 output); the lanes' changed sectors are
// compacted over the warp into `list` (this warp's scratch, 512 entries), then stored 16 sectors per instruction, two
// adjacent lanes per sector, so that each sector is written whole by one store instruction like in stream_vectors.
// The head / tail elements outside the full vectors may share a sector with a neighbouring env: they are written as
// in stream_env, whether they changed or not.
template <typename T>
__device__ __forceinline__ void delta_env(const uint32_t* __restrict__ bits, uint32_t* __restrict__ rec, int bits_words,
                                          int nbits, T* __restrict__ out, int wi, int nw, int lane,
                                          const uint2* __restrict__ lut, uint16_t* __restrict__ list) {
    constexpr int VB = kVecElems<T>, SB = 2 * VB;                     // bits per store vector, per 32-byte sector
    constexpr uint32_t kSectorMask = SB == 32 ? 0xFFFFFFFFu : (1u << SB) - 1u;
    const int pad = obs_pad(out);
    const int total = pad + nbits;
    const int v_begin = (pad + VB - 1) / VB, v_end = total / VB;
    if (wi == 0) stream_edges<T>(bits, nbits, out, v_begin, v_end, lane);
    uint4* vp = reinterpret_cast<uint4*>(out - pad);
    for (int c = wi; 128 * c < bits_words; c += nw) {
        const int wd = 128 * c + 4 * lane;
        uint32_t changed = 0;   // bit j: sector j of this lane's 128 bits differs
        if (wd < bits_words) {
            const uint4 nv = *reinterpret_cast<const uint4*>(bits + wd);
            const uint4 ov = *reinterpret_cast<const uint4*>(rec + wd);
            const uint32_t d[4] = {nv.x ^ ov.x, nv.y ^ ov.y, nv.z ^ ov.z, nv.w ^ ov.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 32 / SB; ++j)
                    if ((d[i] >> (j * SB)) & kSectorMask) changed |= 1u << (i * (32 / SB) + j);
            if (changed) *reinterpret_cast<uint4*>(rec + wd) = nv;
        }
        const int n = __popc(changed);
        int incl = n;   // inclusive prefix sum of n over the warp
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(kFull, incl, o);
            if (lane >= o) incl += t;
        }
        const int n_warp = __shfl_sync(kFull, incl, 31);
        if (n_warp == 0) continue;
        const int s0 = wd * 32 / SB;
        for (int pos = incl - n; changed; changed &= changed - 1u) list[pos++] = (uint16_t)(s0 + __ffs(changed) - 1);
        __syncwarp();
        for (int i = lane >> 1; i < n_warp; i += 16) {
            const int v = 2 * list[i] + (lane & 1);
            if (v >= v_begin && v < v_end) store_vec(vp + v, vector_value<T>(bits, v, lut));
        }
        __syncwarp();
    }
}

// Copies a block's padded bit string into its record (after a full write); warp `wi` of `nw`.
__device__ __forceinline__ void refresh_record(const uint32_t* __restrict__ bits, uint32_t* __restrict__ rec, int bits_words,
                                               int wi, int nw, int lane) {
    for (int i = wi * 32 + lane; i < bits_words / 4; i += nw * 32)
        reinterpret_cast<uint4*>(rec)[i] = reinterpret_cast<const uint4*>(bits)[i];
}

// Packed copy of the observation block for rollout storage: agent a's C*G*G bits start at word a*wpa
// (32x smaller than float32; ctf_unpack_obs expands it again).
__device__ __forceinline__ void store_packed(const DevPlan& P, const uint32_t* __restrict__ bits, int pad,
                                             uint32_t* __restrict__ out_env, int lane) {
    const int CGG = P.C * P.GG, wpa = P.wpa, total = P.N * wpa;
    for (int i = lane; i < total; i += 32) {
        const int a = i / wpa, j = i - a * wpa;
        const int o = pad + a * CGG + 32 * j;
        uint32_t v = __funnelshift_r(bits[o >> 5], bits[(o >> 5) + 1], o & 31);
        const int valid = CGG - 32 * j;            // bits of this word that belong to agent a
        if (valid < 32) v &= (1u << valid) - 1u;
        out_env[i] = v;
    }
}

template <typename T>
__device__ __forceinline__ void write_obs(const DevPlan& P, const Launch& L, const WarpMem& w, long long env, uint32_t me,
                                          uint32_t rev_mask, int lane, const uint2* __restrict__ lut) {
    if (!L.obs && !L.obs_bits) return;
    T* out = L.obs ? reinterpret_cast<T*>(L.obs) + env * (long long)P.E : nullptr;
    const int pad = out ? obs_pad(out) : 0;
    build_obs_bits(P, w, me, rev_mask, pad, lane);
    if (L.obs_bits) store_packed(P, w.bits, pad, L.obs_bits + env * (long long)(P.N * P.wpa), lane);
    if (out) stream_env<T>(w.bits, P.E, out, 0, 1, lane, lut);
    if (out && L.record) {   // a full write into the bound buffer: the record follows it
        refresh_record(w.bits, L.record + env * (long long)P.bits_words, P.bits_words, 0, 1, lane);
        if (lane == 0) L.record_epoch[env] = *L.epoch;
    }
}

// Element codes of the metadata block (host-built, DevPlan::meta_codes): the LANE whose value the element takes.
// write_meta spreads the block's distinct values over the warp — lane i < 8: hp8 of agent i, lane 8 + i: has_flag of
// agent i, lanes 16 / 17 / 18: game progress and the two capture ratios, lane 19: 1.0, lane 20: 0.0 — so that every
// element is one shuffle.
enum : unsigned { kMetaHp = 0, kMetaFlag = 8, kMetaPct = 16, kMetaRatio0 = 17, kMetaRatio1 = 18, kMetaOne = 19, kMetaZero = 20 };

template <bool HPF>
__device__ __forceinline__ void write_meta(const DevPlan& P, uint32_t me, double hpd, int step, int caps0, int caps1,
                                           float* __restrict__ meta_env, int lane) {
    const int N = P.N, M = P.M;
    const int li = lane & 7;
    // hp8[i] = uint8(agent_hp[TYPE_i as agent id] / AGENT_TYPE_HP[TYPE_i])  (:1039-1041)
    const uint32_t src = __shfl_sync(kFull, me, P.meta_hp_src[li]);
    const uint32_t mine = __shfl_sync(kFull, me, li);
    float hp8;
    if (HPF) {   // the same quotient in double, truncated like numpy's float -> uint8 store
        const double srcd = __shfl_sync(kFull, hpd, P.meta_hp_src[li]);
        hp8 = (float)((int)__ddiv_rn(srcd, P.hp_max_f[P.type[li]]) & 0xFF);
    } else {
        hp8 = (float)((ag_hp(src) / P.hp_max_q[P.type[li]]) & 0xFF);
    }
    // the three fp64 quotients that go through float16 (:1035-1036, :1044), one per lane 16..18, in a single pass
    const int num = lane == 16 ? step : (lane == 17 ? caps0 + 1 : caps1 + 1);
    const int den = lane == 16 ? P.game_steps : (lane == 17 ? caps1 + 1 : caps0 + 1);
    const float quot = __half2float(__double2half((double)num / (double)den));
    const float val = lane < 8 ? hp8 : (lane < 16 ? (float)ag_flag(mine) : (lane < 19 ? quot : (lane == 19 ? 1.0f : 0.0f)));
    // The block's layout is static, so the host compiled it into one source lane per element; lane l of pass `it`
    // produces elements 4k .. 4k+3 (k = 32 it + l) and stores them as one float4 (N*M is a multiple of 4 for every N).
    const int n4 = (N * M) >> 2;
    for (int it = 0; it * 32 < n4; ++it) {
        const int k = it * 32 + lane;
        const uint32_t codes = P.meta_codes[k & 63];
        float4 v;
        v.x = __shfl_sync(kFull, val, codes & 31u);
        v.y = __shfl_sync(kFull, val, (codes >> 8) & 31u);
        v.z = __shfl_sync(kFull, val, (codes >> 16) & 31u);
        v.w = __shfl_sync(kFull, val, (codes >> 24) & 31u);
        if (k < n4) reinterpret_cast<float4*>(meta_env)[k] = v;
    }
}

// ------------------------------------------------------------------------------------------------
// State staging
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void store_state(const DevPlan& P, const Launch& L, const WarpMem& w, long long env,
                                            uint32_t me, double hpd, int inv, uint4 ev, int lane) {
    if (P.hp_float && lane < P.N) L.hp[env * P.N + lane] = hpd;
    if (lane < kGridBytes / 16)
        reinterpret_cast<uint4*>(L.grid + env * kGridBytes)[lane] = reinterpret_cast<const uint4*>(w.grid)[lane];
    if (lane < P.N) {
        const unsigned long long rec = (unsigned long long)ag_r(me) | ((unsigned long long)ag_c(me) << 8) |
                                       ((unsigned long long)ag_flag(me) << 16) |
                                       ((unsigned long long)(uint16_t)ag_hp(me) << 32) |
                                       ((unsigned long long)(uint16_t)inv << 48);
        L.agents[env * P.N + lane] = rec;
    }
    if (lane == 0) L.envs[env] = ev;
}

// Per-step counter deltas of this lane's agent, 4 bits per metric (every per-step increment is <= 15:
// at most 4 tags / respawns / neighbours, distances <= GRID_SIZE - 1); added to the HBM counters once per step.
struct Deltas {
    uint32_t lo = 0, hi = 0;  // metrics 0..7, 8..12
};

// Every bump of one actor's turn is warp-uniform (same condition and amount in all lanes), so the turn's deltas are
// summed in uniform registers and merged into the actor's lane once per turn.
template <bool STATS>
__device__ __forceinline__ void bump(Deltas& turn, int metric, uint32_t by) {
    if (STATS) {
        if (metric < 8) turn.lo += by << (4 * metric);
        else turn.hi += by << (4 * (metric - 8));
    }
}

// ------------------------------------------------------------------------------------------------
// reset (gridworld_ctf.py:383-477)
// ------------------------------------------------------------------------------------------------
template <typename T, bool STATS>
__global__ void __launch_bounds__(kThreads) k_reset(const __grid_constant__ DevPlan P, const __grid_constant__ Launch L) {
    extern __shared__ uint4 smem_raw[];
    const uint2* lut = init_expand_lut<T>(smem_raw);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long env = (long long)blockIdx.x * kWarpsPerCta + warp;
    if (env >= L.B) return;
    const WarpMem w = warp_mem(P, reinterpret_cast<unsigned char*>(smem_raw) + kLutBytes<T>, warp);

    if (lane < kGridBytes / 16)
        reinterpret_cast<uint4*>(w.grid)[lane] = reinterpret_cast<const uint4*>(P.grid_template)[lane];
    const int li = lane & 7;
    const uint32_t me = pack_agent(P.start_r[li], P.start_c[li], 0, P.hp_max_q[P.type[li]]);
    const double hpd = P.hp_float ? P.hp_max_f[P.type[li]] : 0.0;
    uint4 ev = make_uint4(0, 0, 0, 0);
    if (!L.first_reset) ev.y = L.envs[env].y + 1;  // episode
    __syncwarp();
    store_state(P, L, w, env, me, hpd, 0, ev, lane);
    if (STATS) {
        const int ns = CTF_N_METRICS * P.N;
        for (int i = lane; i < ns; i += 32) L.stats[env * ns + i] = 0;
        if (L.visits) {
            uint8_t* v = L.visits + env * (long long)P.N * P.GG;
            for (int i = lane; i < P.N * P.GG; i += 32) v[i] = 0;
            __syncwarp();
            if (lane < P.N) v[lane * P.GG + ag_r(me) * P.G + ag_c(me)] = 1;  // update_visitation_map (:473)
        }
    }
    if (L.rewards && lane < P.N) L.rewards[env * P.N + lane] = 0.0f;
    if (L.dones && lane == 0) L.dones[env] = 0;
    const uint32_t rev_mask = (L.rev_override & 0x100u) ? (L.rev_override & 0xFFu)
                                                        : __ballot_sync(kFull, lane < P.N && P.obs_rev[li]);
    if (L.meta) {   // not a hot kernel: the HP representation is a run-time branch here
        if (P.hp_float) write_meta<true>(P, me, hpd, 0, 0, 0, L.meta + env * (long long)P.N * P.M, lane);
        else write_meta<false>(P, me, 0.0, 0, 0, 0, L.meta + env * (long long)P.N * P.M, lane);
    }
    write_obs<T>(P, L, w, env, me, rev_mask, lane, lut);
}

// ------------------------------------------------------------------------------------------------
// observe only
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads) k_observe(const __grid_constant__ DevPlan P, const __grid_constant__ Launch L) {
    extern __shared__ uint4 smem_raw[];
    const uint2* lut = init_expand_lut<T>(smem_raw);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long env = (long long)blockIdx.x * kWarpsPerCta + warp;
    if (env >= L.B) return;
    const WarpMem w = warp_mem(P, reinterpret_cast<unsigned char*>(smem_raw) + kLutBytes<T>, warp);
    if (lane < kGridBytes / 16)
        reinterpret_cast<uint4*>(w.grid)[lane] = reinterpret_cast<const uint4*>(L.grid + env * kGridBytes)[lane];
    const int li = lane & 7;
    uint32_t me = 0;
    double hpd = 0.0;
    if (lane < P.N) {
        const unsigned long long rec = L.agents[env * P.N + lane];
        me = pack_agent((int)(rec & 0xFF), (int)((rec >> 8) & 0xFF), (int)((rec >> 16) & 1), (int)(short)(rec >> 32));
        if (P.hp_float) hpd = L.hp[env * P.N + lane];
    }
    const uint4 ev = L.envs[env];
    __syncwarp();
    const uint32_t rev_mask = (L.rev_override & 0x100u) ? (L.rev_override & 0xFFu)
                                                        : __ballot_sync(kFull, lane < P.N && P.obs_rev[li]);
    if (L.meta) {
        if (P.hp_float) write_meta<true>(P, me, hpd, (int)ev.x, (int)ev.z, (int)ev.w, L.meta + env * (long long)P.N * P.M, lane);
        else write_meta<false>(P, me, 0.0, (int)ev.x, (int)ev.z, (int)ev.w, L.meta + env * (long long)P.N * P.M, lane);
    }
    write_obs<T>(P, L, w, env, me, rev_mask, lane, lut);
}

// ------------------------------------------------------------------------------------------------
// step (gridworld_ctf.py:849-918) + observations for every agent
// ------------------------------------------------------------------------------------------------
// One env step by one warp: state in, act / tag / respawn / heal / rewards / statistics / metadata, state out.
// Returns the lane's agent register (position for the observation's self plane) and the per-agent reverse_grid mask;
// the tile map of the new state is left in w.grid for the observation writer.
// HPF: HP is an IEEE double per agent (plan.hp_float) instead of the fixed-point field of the agent register; every
// operation on it is the reference's Python float operation (:648-650 vault gate, :656 vault cost, :818 damage, :824
// lethal test, :785 respawn, :845-846 heal), so non-dyadic HP configurations stay bit-exact.
template <bool STATS, bool HPF>
__device__ __forceinline__ uint32_t step_env(const DevPlan& P, const Launch& L, const WarpMem& w, long long env, int lane,
                                             uint32_t& rev_mask_out) {
    const int N = P.N;
    const int li = lane & 7;

    // ---- stage state: tile map -> shared memory, agent i -> lane i
    if (lane < kGridBytes / 16)
        reinterpret_cast<uint4*>(w.grid)[lane] = reinterpret_cast<const uint4*>(L.grid + env * kGridBytes)[lane];
    uint32_t me = 0;
    int inv = 0;
    int action = 4;
    if (lane < N) {
        const unsigned long long rec = L.agents[env * N + lane];
        me = pack_agent((int)(rec & 0xFF), (int)((rec >> 8) & 0xFF), (int)((rec >> 16) & 1), (int)(short)(rec >> 32));
        inv = (int)((rec >> 48) & 0xFFFF);
        action = L.actions[env * N + lane];
    }
    uint4 ev = L.envs[env];
    double hpd = 0.0;   // this lane's agent's HP (HPF only; dead code otherwise)
    if (HPF && lane < N) hpd = L.hp[env * N + lane];
    Deltas dl;
    const int my_team = P.team[li], my_type = P.type[li], my_slot = P.my_slot[li];
    const bool bad_action = lane < N && action >= CTF_N_ACTIONS;
    if (__any_sync(kFull, bad_action)) {
        if (lane == 0) atomicOr(L.faults, CTF_FAULT_BAD_ACTION);
        if (bad_action) action = 4;
    }
    if (P.reverse_team1_actions && my_team == 1) action = P.rev_action[action];

    // ---- step counter and this step's draws: lane l generates site l
    ev.x += 1;                                  // env_step_count += 1 (:857)
    const int step = (int)ev.x;
    uint32_t wd[4];
    philox4x32_10(L.env_id_base + (uint32_t)env, ev.y, ev.x, (uint32_t)lane, L.seed_lo, L.seed_hi, wd);

    // ---- move order: Fisher-Yates from the identity with word 2 of site i (dice_roll :734-742)
    uint32_t order = 0x76543210u;
    for (int i = N - 1; i >= 1; --i) {
        const uint32_t wi = __shfl_sync(kFull, wd[2], i);
        const int j = (int)__umulhi(wi, (uint32_t)(i + 1));
        const uint32_t x = ((order >> (4 * i)) ^ (order >> (4 * j))) & 15u;
        order ^= (x << (4 * i)) | (x << (4 * j));
    }
    __syncwarp();

    uint32_t turn_pos = 0;      // this lane's agent's position at the end of its own turn (zonal metrics)
    bool captured = false;      // this lane's agent captured during its own act (:728-730)
    bool tag_reward = false;    // this lane's agent made a lethal tag (:832)
    uint32_t cap_team = 0;      // _flag_capture_team_current_move as bits (:858)
    int caps0 = (int)ev.z, caps1 = (int)ev.w;

    for (int s = 0; s < N; ++s) {
        const int a = (order >> (4 * s)) & 15;                 // acting agent (warp-uniform)
        const uint32_t am = __shfl_sync(kFull, me, a);
        const int act_code = __shfl_sync(kFull, action, a);
        const int type = P.type[a], team = P.team[a], tile = P.tile[a];
        int ar = ag_r(am), ac = ag_c(am), aflag = ag_flag(am), ahp = ag_hp(am);
        int ainv = (type == 3) ? __shfl_sync(kFull, inv, a) : 0;
        double ahpd = HPF ? __shfl_sync(kFull, hpd, a) : 0.0;
        bool cap_now = false;
        Deltas turn;                                           // this turn's counter increments (warp-uniform)

        // ---------------- act (:700-732)
        const int nr = ar + P.delta[type][act_code][0], nc = ac + P.delta[type][act_code][1];
        if (nr >= 0 && nr < P.G && nc >= 0 && nc < P.G) {     // is_valid_move (:636-641)
            const int target = w.grid[nr * kRow + nc];
            const bool can_vault = HPF ? (__dsub_rn(ahpd, P.vault_cost_f) > P.vault_min_f) : ((ahp - P.vault_cost_q) > P.vault_min_q);
            if (target == 0 && (act_code <= 3 || (act_code >= 5 && type == 2 && can_vault))) {
                // movement_handler (:569-612); every lane stores the same bytes
                __syncwarp();
                w.grid[ar * kRow + ac] = 0;
                w.grid[nr * kRow + nc] = (uint8_t)tile;
                __syncwarp();
                ar = nr; ac = nc;
                const int ofr = P.flag_pos[1 - team][0], ofc = P.flag_pos[1 - team][1];
                const int hfr = P.flag_pos[team][0], hfc = P.flag_pos[team][1];
                if (cheb(nr, nc, ofr, ofc) <= 1 && w.grid[ofr * kRow + ofc] == P.flag_tile[1 - team]) {  // pickup (:583-591)
                    aflag = 1;
                    __syncwarp();
                    w.grid[ofr * kRow + ofc] = 1;
                    __syncwarp();
                    bump<STATS>(turn, CTF_M_FLAG_PICKUPS, 1);
                }
                if (cheb(nr, nc, hfr, hfc) <= 1 && aflag == 1 &&
                    (!P.home_flag_capture || w.grid[hfr * kRow + hfc] == P.flag_tile[team])) {        // capture (:594-610)
                    aflag = 0;
                    __syncwarp();
                    w.grid[ofr * kRow + ofc] = P.flag_tile[1 - team];
                    __syncwarp();
                    if (team == 0) caps0 += 1; else caps1 += 1;
                    cap_team |= 1u << team;
                    cap_now = true;
                    bump<STATS>(turn, CTF_M_FLAG_CAPTURES, 1);
                }
                if (act_code >= 5 && type == 2) {                                                   // (:652-657)
                    if (HPF) ahpd = __dsub_rn(ahpd, P.vault_cost_f);
                    else ahp -= P.vault_cost_q;
                }
            } else if (act_code >= 5 && type == 3 && ainv > 0 && target == 0 &&
                       cheb(nr, nc, P.spawn_pos[team][0], P.spawn_pos[team][1]) > 1 &&
                       cheb(nr, nc, P.spawn_pos[1 - team][0], P.spawn_pos[1 - team][1]) > 1) {
                // add_block (:614-634)
                __syncwarp();
                w.grid[nr * kRow + nc] = 2;
                __syncwarp();
                ainv -= 1;
                if (STATS) {
                    bump<STATS>(turn, CTF_M_BLOCKS_LAID, 1);
                    bump<STATS>(turn, CTF_M_BLOCKS_LAID_DIST_OWN_FLAG, (uint32_t)cheb(ar, ac, P.capture_pos[team][0], P.capture_pos[team][1]));
                    bump<STATS>(turn, CTF_M_BLOCKS_LAID_DIST_OPP_FLAG, (uint32_t)cheb(ar, ac, P.capture_pos[1 - team][0], P.capture_pos[1 - team][1]));
                }
            } else if (act_code < 5 && type == 3 && (target == 2 || target == 3)) {
                // mine_block (:677-690)
                __syncwarp();
                w.grid[nr * kRow + nc] = (target == 2) ? 3 : 0;
                __syncwarp();
                if (target == 3) {
                    if (ainv < P.max_agent_blocks) ainv += P.block_pickup_value;
                    bump<STATS>(turn, CTF_M_BLOCKS_MINED, 1);
                }
            }
        }
        if (lane == a) {
            me = pack_agent(ar, ac, aflag, ahp);
            if (HPF) hpd = ahpd;
            inv = ainv;
            captured = cap_now;
        }

        // distance of this lane's agent to the actor after its move: tag range now, adjacency metrics below
        // (recomputed there only if a respawn moved somebody in between)
        const int d_me = cheb(ar, ac, ag_r(me), ag_c(me));
        bool moved_by_respawn = false;

        // ---------------- tagging_logic (:796-837)
        if (HPF ? (P.damage_f[type] > 0.0) : (P.damage_q[type] > 0)) {
            const bool boosted = type == 1 && cheb(ar, ac, P.flag_pos[team][0], P.flag_pos[team][1]) <= P.guardian_distance;
            const int dmg = boosted ? P.damage_boosted_q[type] : P.damage_q[type];
            const double dmgd = HPF ? (boosted ? P.damage_boosted_f[type] : P.damage_f[type]) : 0.0;
            const bool is_opp = lane < N && my_team != team && my_slot >= 0;
            const int site = 4 * a + (my_slot < 0 ? 0 : my_slot);
            const uint32_t roll = __shfl_sync(kFull, wd[0], site);
            const uint32_t pick_word = __shfl_sync(kFull, wd[1], site);
            const bool hit = is_opp && (unsigned long long)roll < P.tag_threshold && d_me <= P.tagging_range;
            int hp = ag_hp(me);
            if (hit) hp -= dmg;                                                                      // (:818)
            if (HPF && hit) hpd = __dsub_rn(hpd, dmgd);
            const bool lethal = hit && (HPF ? (hpd <= 0.0) : (hp <= 0));                             // (:824)
            if (!HPF && hit) me = (me & 0xFFFFu) | ((uint32_t)(hp & 0xFFFF) << 16);
            const unsigned hits = __ballot_sync(kFull, hit);
            unsigned deaths = __ballot_sync(kFull, lethal);
            moved_by_respawn = deaths != 0;
            if (STATS && hits) bump<STATS>(turn, CTF_M_TAG_COUNT, (uint32_t)__popc(hits));
            // lethal hits respawn one after the other in opponent-id order: each changes the next one's window
            while (deaths) {
                const int opp = __ffs(deaths) - 1;
                deaths &= deaths - 1;
                const uint32_t om = __shfl_sync(kFull, me, opp);
                const uint32_t ow = __shfl_sync(kFull, pick_word, opp);
                const int oteam = 1 - team;
                if (ag_flag(om)) bump<STATS>(turn, CTF_M_FLAG_DISPOSSESSIONS, 1);
                // respawn (:761-794): open cells of the clipped 3x3 window around the victim's spawn, row-major
                const int x = P.spawn_pos[oteam][0], y = P.spawn_pos[oteam][1];
                const int wr = x - 1 + lane / 3, wc = y - 1 + lane % 3;
                const bool open = lane < 9 && wr >= 0 && wr < P.G && wc >= 0 && wc < P.G && w.grid[wr * kRow + wc] == 0;
                const unsigned cand = __ballot_sync(kFull, open);
                const int k = __popc(cand);
                if (k > 0) {
                    const int pick = (int)__umulhi(ow, (uint32_t)k);                                 // randint(k) (:771)
                    const int bit = __fns(cand, 0, pick + 1);
                    const int rr = x - 1 + bit / 3, rc = y - 1 + bit % 3;
                    const int old_r = ag_r(om), old_c = ag_c(om);
                    __syncwarp();
                    w.grid[old_r * kRow + old_c] = 0;
                    w.grid[rr * kRow + rc] = P.tile[opp];
                    if (ag_flag(om)) {                                                                // (:788-794)
                        if (P.drop_flag_when_no_hp) w.grid[old_r * kRow + old_c] = P.flag_tile[1 - oteam];
                        else w.grid[P.flag_pos[1 - oteam][0] * kRow + P.flag_pos[1 - oteam][1]] = P.flag_tile[1 - oteam];
                    }
                    __syncwarp();
                    if (lane == opp) {
                        me = pack_agent(rr, rc, 0, HPF ? 0 : P.hp_max_q[P.type[opp]]);
                        if (HPF) hpd = P.hp_max_f[P.type[opp]];                                       // (:785)
                    }
                } else if (lane == 0) {
                    atomicOr(L.faults, CTF_FAULT_RESPAWN_BLOCKED);   // randint(0) raises in the reference (:771)
                }
                if (lane == a) tag_reward = true;
                bump<STATS>(turn, CTF_M_RESPAWN_TAG_COUNT, 1);
            }
        }

        // ---------------- proximity metrics (:890-902); the zonal ones (:879-889) only need the actor's position at
        // its own turn, which lane a keeps in turn_pos: they are evaluated for all agents at once after the loop
        if (STATS) {
            if (lane == a) turn_pos = (uint32_t)ar | ((uint32_t)ac << 4);
            const int d_now = moved_by_respawn ? cheb(ar, ac, ag_r(me), ag_c(me)) : d_me;
            const bool near = lane < N && my_slot >= 0 && d_now <= 1;
            const unsigned mates = __ballot_sync(kFull, near && my_team == team);   // includes the agent itself
            const unsigned opps = __ballot_sync(kFull, near && my_team != team);
            if (mates) bump<STATS>(turn, CTF_M_STEPS_ADJ_TEAMMATE, (uint32_t)__popc(mates));
            if (opps) bump<STATS>(turn, CTF_M_STEPS_ADJ_OPPONENT, (uint32_t)__popc(opps));
            if (lane == a) { dl.lo += turn.lo; dl.hi += turn.hi; }
        }
    }

    // ---- zonal metrics (:879-889) of every agent, at the position it had at its own turn
    if (STATS) {
        const int tr = (int)(turn_pos & 15u), tc = (int)(turn_pos >> 4);
        const int d_own = cheb(tr, tc, P.capture_pos[my_team][0], P.capture_pos[my_team][1]);
        const int d_opp = cheb(tr, tc, P.capture_pos[1 - my_team][0], P.capture_pos[1 - my_team][1]);
        dl.hi += ((d_own <= P.zone_distance ? 1u : 0u) << (4 * (CTF_M_STEPS_DEFENDING_ZONE - 8))) +
                 ((d_opp <= P.zone_distance ? 1u : 0u) << (4 * (CTF_M_STEPS_ATTACKING_ZONE - 8)));
    }
    // ---- heal_agents (:839-847)
    {
        if (HPF) {
            const double mxd = P.hp_max_f[my_type];
            if (hpd < mxd) hpd = fmin(__dadd_rn(hpd, P.heal_f), mxd);
        } else {
            const int mx = P.hp_max_q[my_type];
            int hp = ag_hp(me);
            if (hp < mx) hp = min(hp + P.heal_q, mx);
            me = (me & 0xFFFFu) | ((uint32_t)(hp & 0xFFFF) << 16);
        }
    }
    // ---- rewards (:727-730, :873, :957-966, :920-940) in fp64, stored as fp32 (ppo.py:108)
    const bool done = step >= P.game_steps;   // set at step == GAME_STEPS and never cleared until reset (:914-915)
    {
        // every operation is a separately rounded IEEE add / multiply (__dadd_rn / __dmul_rn are never contracted
        // into an FMA): -0.5 + 5 * 0.1 must give the reference's exact 0.0, not the fused 2.8e-17
        double r = 0.0;
        r = __dadd_rn(r, P.reward_step);
        if (captured) r = __dadd_rn(r, P.reward_capture);
        if (tag_reward) r = __dadd_rn(r, P.reward_tag);
        if (P.use_adjusted_rewards && ((cap_team >> (1 - my_team)) & 1u)) r = __dadd_rn(r, -P.capture_punish);
        if (step == P.game_steps && caps0 != caps1) {
            const double margin = (double)abs(caps0 - caps1);
            const int winner = caps0 > caps1 ? 0 : 1;
            if (my_team == winner) r = __dadd_rn(r, __dmul_rn(margin, P.win_margin));
            else r = __dadd_rn(r, -__dmul_rn(margin, P.loss_margin));
        }
        if (L.rewards && lane < N) L.rewards[env * N + lane] = (float)r;
    }
    if (L.dones && lane == 0) L.dones[env] = done ? 1 : 0;
    ev.z = (uint32_t)caps0;
    ev.w = (uint32_t)caps1;

    // ---- write state back
    __syncwarp();
    store_state(P, L, w, env, me, hpd, inv, ev, lane);
    if (STATS) {
        if (lane < N) {   // fire-and-forget reductions: no load latency, nothing held in registers
            uint32_t* sp = L.stats + env * (long long)(CTF_N_METRICS * N) + lane;
#pragma unroll
            for (int m = 0; m < CTF_N_METRICS; ++m) {
                const uint32_t v = ((m < 8 ? dl.lo : dl.hi) >> (4 * (m & 7))) & 15u;
                if (v) atomicAdd(sp + m * N, v);
            }
        }
        if (L.visits && lane < N) {   // update_visitation_map (:911), uint8 wrap
            uint8_t* v = L.visits + (env * N + lane) * (long long)P.GG + ag_r(me) * P.G + ag_c(me);
            *v = (uint8_t)(*v + 1);
        }
    }

    rev_mask_out = (L.rev_override & 0x100u) ? (L.rev_override & 0xFFu) : __ballot_sync(kFull, lane < N && P.obs_rev[li]);
    if (L.meta) write_meta<HPF>(P, me, hpd, step, caps0, caps1, L.meta + env * (long long)N * P.M, lane);
    return me;
}

// Warp-per-env step kernel of ctf_step: every warp steps its env and builds that env's observation
// bit string in its own shared-memory buffer; after one barrier the CTA's warps write the CTA's kWarpsPerCta consecutive
// env blocks one after the other, all warps on the same block (2 KB contiguous per pass) — a quarter as many open
// write streams as when every warp streams its own block, and each CTA's region goes out in address order.
// profiles/r02_coop_stream.log: 8_arena float32 0.980 -> 0.974 ms, uint8 0.283 -> 0.281, 7_gridlocked B = 16384 0.1475 -> 0.1450;
// 4 warps x 5 resident CTAs and 2 x 9 tie, 8 x 3 (0.987) and 16 x 1 (1.18) lose: the barrier idles too much of the SM.
// Per-env ready flags instead of the barrier (a block is written by whichever warps are ready) are SLOWER, 0.9825 vs 0.9786 ms,
// uint8 0.295 vs 0.2835 (profiles/r02_coop_flag.log): the aligned passes are what helps.
//
// With a record bound to L.obs (ctf_bind_obs_record) an env whose record is valid (its epoch is the current one) is
// written as a delta (delta_env): only the ~1.3 % of sectors that changed since the last write.  An env whose record
// is not valid is written in full by stream_env, its record copied from the string and stamped.  Each warp decides for
// its own env before the barrier, so that no warp of the CTA reads an epoch another warp has already stamped.
// DELTA (L.record set) is a template parameter: the launches without a record run the code they ran before the record
// existed (uint8, packed-only and the step logic itself lost 11-15 % when one kernel carried both paths).
template <typename T, bool STATS, bool HPF, bool DELTA>
__global__ void __launch_bounds__(kThreads) k_step(const __grid_constant__ DevPlan P, const __grid_constant__ Launch L) {
    extern __shared__ uint4 smem_raw[];
    __shared__ int s_full[DELTA ? kWarpsPerCta : 1];   // env e of the CTA is written in full
    const uint2* lut = init_expand_lut<T>(smem_raw);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long env = (long long)blockIdx.x * kWarpsPerCta + warp;
    unsigned char* base = reinterpret_cast<unsigned char*>(smem_raw) + kLutBytes<T>;
    if (env < L.B) {
        const WarpMem w = warp_mem(P, base, warp);
        uint32_t* rec = DELTA ? L.record + env * (long long)P.bits_words : nullptr;
        // the old record is read after the barrier: start moving it into L2 while the env steps
        if (DELTA && lane * 32 < P.bits_words) asm volatile("prefetch.global.L2 [%0];" ::"l"(rec + lane * 32));
        uint32_t rev_mask;
        const uint32_t me = step_env<STATS, HPF>(P, L, w, env, lane, rev_mask);
        if (L.obs || L.obs_bits) {
            T* out = L.obs ? reinterpret_cast<T*>(L.obs) + env * (long long)P.E : nullptr;
            const int pad = out ? obs_pad(out) : 0;
            build_obs_bits(P, w, me, rev_mask, pad, lane);
            if (L.obs_bits) store_packed(P, w.bits, pad, L.obs_bits + env * (long long)(P.N * P.wpa), lane);
        }
        if (DELTA && lane == 0) {
            const uint32_t ep = *L.epoch;
            const bool full = L.record_epoch[env] != ep;
            if (full) L.record_epoch[env] = ep;
            s_full[warp] = full;
        }
    }
    __syncthreads();
    if (L.obs) {
        for (int e = 0; e < kWarpsPerCta; ++e) {
            const long long env_e = (long long)blockIdx.x * kWarpsPerCta + e;
            if (env_e >= L.B) break;
            const uint32_t* bits = warp_mem(P, base, e).bits;
            T* out = reinterpret_cast<T*>(L.obs) + env_e * (long long)P.E;
            if (DELTA) {
                uint32_t* rec = L.record + env_e * (long long)P.bits_words;
                if (!s_full[e]) {
                    delta_env<T>(bits, rec, P.bits_words, P.E, out, warp, kWarpsPerCta, lane, lut,
                                 reinterpret_cast<uint16_t*>(warp_mem(P, base, warp).list));
                } else {
                    stream_env<T>(bits, P.E, out, warp, kWarpsPerCta, lane, lut);
                    refresh_record(bits, rec, P.bits_words, warp, kWarpsPerCta, lane);
                }
            } else {
                stream_env<T>(bits, P.E, out, warp, kWarpsPerCta, lane, lut);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// packed observations -> policy input: one CTA per chunk of consecutive agent blocks
// ------------------------------------------------------------------------------------------------
// The chunk's packed words (wpa per block, coalesced) are re-packed in shared memory into ONE contiguous bit string
// (block b's nbits elements follow block b-1's directly, shifted by the output's alignment pad) and all warps stream
// the chunk's output region together — CTAs are scheduled in address order, so few blocks are open at a time.
constexpr int kUnpackThreads = 256;   // 512 measured too: profiles/r02_unpack_threads.log
template <typename T>
__global__ void __launch_bounds__(kUnpackThreads) k_unpack(const uint32_t* __restrict__ packed, T* __restrict__ out,
                                                          long long n_blocks, int nbits, int wpa, int chunk, int bits_words) {
    extern __shared__ uint4 smem_raw[];
    const uint2* lut = init_expand_lut<T>(smem_raw);
    uint32_t* bits = reinterpret_cast<uint32_t*>(reinterpret_cast<unsigned char*>(smem_raw) + kLutBytes<T>);   // [bits_words]
    uint32_t* pk = bits + bits_words;                          // [chunk * wpa]
    const long long blk0 = (long long)blockIdx.x * chunk;
    const int nb = (int)min((long long)chunk, n_blocks - blk0);
    if (nb <= 0) return;
    for (int i = threadIdx.x; i < nb * wpa; i += kUnpackThreads) pk[i] = __ldg(packed + blk0 * wpa + i);
    __syncthreads();
    T* dst = out + blk0 * (long long)nbits;
    const int pad = obs_pad(dst), total = nb * nbits;
    for (int wd = threadIdx.x; wd < bits_words; wd += kUnpackThreads) {
        uint32_t val = 0;
        int k = 0, e = 32 * wd - pad;              // bit k of this word is element e + k of the chunk
        if (e < 0) { k = -e; e = 0; }
        while (k < 32 && e < total) {
            const int b = e / nbits, o = e - b * nbits, j = o >> 5;
            const int take = min(32 - k, nbits - o);
            const uint32_t lo = pk[b * wpa + j], hi = j + 1 < wpa ? pk[b * wpa + j + 1] : 0u;
            uint32_t v = __funnelshift_r(lo, hi, o & 31);
            if (take < 32) v &= (1u << take) - 1u;
            val |= v << k;
            k += take; e += take;
        }
        bits[wd] = val;
    }
    __syncthreads();
    stream_env<T>(bits, total, dst, threadIdx.x >> 5, kUnpackThreads / 32, threadIdx.x & 31, lut);
}

// ------------------------------------------------------------------------------------------------
// per-handle sum of the per-env counters
// ------------------------------------------------------------------------------------------------
__global__ void k_stats_sum(const uint32_t* __restrict__ stats, long long B, int ns, unsigned long long* __restrict__ out) {
    // thread t handles counter (t % ns) of envs blockIdx.x*chunk + ...; consecutive threads read consecutive words
    const long long chunk = (B + gridDim.x - 1) / gridDim.x;
    const long long b0 = blockIdx.x * chunk, b1 = min(B, b0 + chunk);
    const int per_pass = blockDim.x / ns;       // envs handled concurrently by this block
    const int sub = threadIdx.x / ns, k = threadIdx.x % ns;
    if (sub >= per_pass) return;
    unsigned long long acc = 0;
    for (long long b = b0 + sub; b < b1; b += per_pass) acc += stats[b * ns + k];
    if (acc) atomicAdd(&out[k], acc);
}

// ------------------------------------------------------------------------------------------------
// policy trunk from packed observations: conv1 (sparse, fp32) -> tanh -> conv2 (mma.sync bf16) -> tanh -> fc1 input rows
// ------------------------------------------------------------------------------------------------
// One warp owns one sample at a time; the CTA's warps share the conv weights in shared memory.
// Per sample: the wpa packed words are staged, a per-cell channel mask is built from them, conv1 accumulates for every
// output position the bias plus the weight columns of the set (cell, channel) pairs of its 3x3 window (exact for any
// {0,1} input; cost grows with the number of set bits), and stores tanh as bf16 in a [position][16 channels] tile.
// conv2 is an implicit GEMM on that tile: M = (G-4)^2 positions, N = 32 channels, K = 9 taps x 16 channels, one
// m16n8k16 k-step per tap.  The epilogue writes one n-tile (8 channels = a contiguous 8*(G-4)^2 run of the (c, y, x)
// feature row) at a time through shared memory so that the row is written with 16-byte stores.
constexpr int kTrunkWarps = 8;
constexpr int kTrunkThreads = kTrunkWarps * 32;
constexpr int kTrunkW2Words = 9 * 4 * 32 * 2;   // conv2 B fragments: [tap][n-tile][lane][2 x bf16x2]

// what every trunk launch reads, whatever its policies and segments: shapes, shared-memory layout, inputs and output
struct TrunkGeometry {
    const uint32_t* packed;
    const float* meta;
    __nv_bfloat16* features;
    long long stride;
    int ape;
    int G, C, GG, wpa, M;
    int S1, S2;              // conv1 / conv2 output side
    int warp_words;          // shared-memory words per warp
    int off_mask, off_act, off_stage;   // word offsets inside a warp's region
};

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&v);
}

// Channel mask of every cell, then conv1 -> tanh -> bf16 of one sample into act ([S1*S1][8] bf16x2): the part of the
// trunk that k_policy_trunk computes and k_policy_trunk_backward recomputes bit for bit.  Cells and positions first,
// first + step, ...: the forward's warp passes (lane, 32, __syncwarp), the backward's CTA (thread, CTA size,
// __syncthreads).  conv1 adds, for every output position, the bias plus the weight columns of the set (cell, channel)
// pairs of its 3x3 window in a fixed order (dy, dx, c ascending).
template <typename Sync>
__device__ __forceinline__ void trunk_conv1(const uint32_t* bits, uint16_t* cmask, uint32_t* act, const float* w1,
                                            const float* b1, int C, int G, int GG, int S1, int first, int step, Sync sync) {
    // channel mask of every cell: bit c = element c*GG + p
    for (int p = first; p < GG; p += step) {
        uint32_t m = 0;
        for (int c = 0; c < C; ++c) {
            const int el = c * GG + p;
            m |= ((bits[el >> 5] >> (el & 31)) & 1u) << c;
        }
        cmask[p] = (uint16_t)m;
    }
    sync();
    for (int q = first; q < S1 * S1; q += step) {
        const int y = q / S1, x = q - y * S1;
        float acc[16];
#pragma unroll
        for (int o = 0; o < 16; ++o) acc[o] = b1[o];
        for (int dy = 0; dy < 3; ++dy) {
            for (int dx = 0; dx < 3; ++dx) {
                uint32_t m = cmask[(y + dy) * G + x + dx];
                while (m) {
                    const int c = __ffs(m) - 1;
                    m &= m - 1;
                    const float4* col = reinterpret_cast<const float4*>(w1 + ((c * 3 + dy) * 3 + dx) * 16);
#pragma unroll
                    for (int v = 0; v < 4; ++v) {
                        const float4 wv = col[v];
                        acc[4 * v] += wv.x; acc[4 * v + 1] += wv.y; acc[4 * v + 2] += wv.z; acc[4 * v + 3] += wv.w;
                    }
                }
            }
        }
        uint4 lo, hi;
        lo.x = pack_bf16x2(tanhf(acc[0]), tanhf(acc[1]));   lo.y = pack_bf16x2(tanhf(acc[2]), tanhf(acc[3]));
        lo.z = pack_bf16x2(tanhf(acc[4]), tanhf(acc[5]));   lo.w = pack_bf16x2(tanhf(acc[6]), tanhf(acc[7]));
        hi.x = pack_bf16x2(tanhf(acc[8]), tanhf(acc[9]));   hi.y = pack_bf16x2(tanhf(acc[10]), tanhf(acc[11]));
        hi.z = pack_bf16x2(tanhf(acc[12]), tanhf(acc[13])); hi.w = pack_bf16x2(tanhf(acc[14]), tanhf(acc[15]));
        reinterpret_cast<uint4*>(act)[2 * q] = lo;
        reinterpret_cast<uint4*>(act)[2 * q + 1] = hi;
    }
}

// Copies one policy's conv weights into the CTA's shared memory for k_policy_trunk: conv1 as [C*9][16] columns, the
// biases, the conv2 B fragments.  The caller synchronises the CTA after it, and before it when other warps may still
// read the previous policy's weights.
__device__ __forceinline__ void trunk_stage_weights(const float* conv1_w, const float* conv1_b, const uint2* conv2_w,
                                                    const float* conv2_b, int C, float* w1, float* b1, float* b2, uint2* w2) {
    for (int i = threadIdx.x; i < C * 9 * 16; i += kTrunkThreads) {
        const int o = i & 15, tap = i >> 4;                              // tap = c*9 + dy*3 + dx
        w1[i] = conv1_w[o * C * 9 + tap];
    }
    if (threadIdx.x < 16) b1[threadIdx.x] = conv1_b[threadIdx.x];
    if (threadIdx.x < 32) b2[threadIdx.x] = conv2_b[threadIdx.x];
    for (int i = threadIdx.x; i < kTrunkW2Words / 2; i += kTrunkThreads) w2[i] = conv2_w[i];
}

// One sample of the trunk, computed by one warp with the weights staged in shared memory: stages packed block `blk`
// (A.packed, A.wpa words), conv1 (trunk_conv1), conv2 on tensor cores, tanh, bf16, then the metadata row `blk` and
// zeros up to A.stride, into feature row `r` of A.features.
__device__ __forceinline__ void trunk_sample(const TrunkGeometry& A, long long blk, long long r, const float* w1,
                                             const float* b1, const float* b2, const uint2* w2, uint32_t* bits,
                                             uint16_t* cmask, uint32_t* act, __nv_bfloat16* stage, int lane, int C, int G,
                                             int GG, int S1, int S2, int M2, int g, int t, int n_mt, long long conv_elems) {
    const uint32_t* src = A.packed + blk * A.wpa;
    for (int i = lane; i < A.wpa; i += 32) bits[i] = __ldg(src + i);
    __syncwarp();
    trunk_conv1(bits, cmask, act, w1, b1, C, G, GG, S1, lane, 32, [] { __syncwarp(); });
    __syncwarp();
    __nv_bfloat16* row = A.features + r * A.stride;
    // conv2: n-tile (8 output channels) outer, m-tile (16 positions) inner, one k-step per tap
    for (int nt = 0; nt < 4; ++nt) {
        const float bias0 = b2[8 * nt + 2 * t], bias1 = b2[8 * nt + 2 * t + 1];
        for (int mt = 0; mt < n_mt; ++mt) {
            const int m0 = min(mt * 16 + g, M2 - 1), m1 = min(mt * 16 + g + 8, M2 - 1);   // pad rows: any valid position
            const int y0 = m0 / S2, y1 = m1 / S2;
            const int p0 = y0 * S1 + (m0 - y0 * S2), p1 = y1 * S1 + (m1 - y1 * S2);
            float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
                const int off = (tap / 3) * S1 + (tap % 3);
                const uint32_t a0 = act[(p0 + off) * 8 + t], a1 = act[(p1 + off) * 8 + t];
                const uint32_t a2 = act[(p0 + off) * 8 + t + 4], a3 = act[(p1 + off) * 8 + t + 4];
                const uint2 b = w2[(tap * 4 + nt) * 32 + lane];
                asm volatile(
                    "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
                    "{%0,%1,%2,%3};\n"
                    : "+f"(d0), "+f"(d1), "+f"(d2), "+f"(d3)
                    : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b.x), "r"(b.y));
            }
            const int r0 = mt * 16 + g, r1 = r0 + 8;
            if (r0 < M2) {
                stage[(2 * t) * M2 + r0] = __float2bfloat16_rn(tanhf(d0 + bias0));
                stage[(2 * t + 1) * M2 + r0] = __float2bfloat16_rn(tanhf(d1 + bias1));
            }
            if (r1 < M2) {
                stage[(2 * t) * M2 + r1] = __float2bfloat16_rn(tanhf(d2 + bias0));
                stage[(2 * t + 1) * M2 + r1] = __float2bfloat16_rn(tanhf(d3 + bias1));
            }
        }
        __syncwarp();
        // channels 8nt .. 8nt+7 are elements [8nt*M2, 8(nt+1)*M2) of the row: 16*M2 bytes, 16-byte aligned
        uint4* dst = reinterpret_cast<uint4*>(row + (long long)8 * nt * M2);
        const uint4* sv = reinterpret_cast<const uint4*>(stage);
        for (int i = lane; i < M2; i += 32) dst[i] = sv[i];
        __syncwarp();
    }
    // metadata as bf16, then zeros up to the stride (8 elements per 16-byte store)
    const float* mrow = A.meta + blk * A.M;
    const int tail = (int)((A.stride - conv_elems) >> 3);
    uint4* dst = reinterpret_cast<uint4*>(row + conv_elems);
    for (int i = lane; i < tail; i += 32) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int c = 8 * i + u;
            v[u] = c < A.M ? __ldg(mrow + c) : 0.f;
        }
        dst[i] = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
    }
    __syncwarp();
}

// shared-memory layout of k_policy_trunk for a plan: bytes of the CTA-wide weights, words per warp and the offsets
static __host__ void trunk_layout(const DevPlan& P, TrunkGeometry& A, size_t& smem) {
    const int S1 = P.G - 2, S2 = P.G - 4;
    const auto up4 = [](int w) { return (w + 3) & ~3; };                 // 16-byte alignment in words
    A.G = P.G; A.C = P.C; A.GG = P.GG; A.wpa = P.wpa; A.M = P.M; A.S1 = S1; A.S2 = S2;
    A.off_mask = up4(P.wpa);
    A.off_act = A.off_mask + up4((P.GG + 1) / 2);
    A.off_stage = A.off_act + S1 * S1 * 8;
    A.warp_words = A.off_stage + up4(4 * S2 * S2);                       // 8 channels x S2^2 bf16
    const size_t shared_words = (size_t)P.C * 9 * 16 + 16 + 32 + kTrunkW2Words;
    smem = (shared_words + (size_t)kTrunkWarps * A.warp_words) * 4;
}

// One launch computes the samples of one or more (policy, env range, agent ids) segments.  The segments' samples are
// cut into tiles of kTrunkWarps consecutive samples of one segment (a segment's last tile may be shorter); the host
// numbers the tiles in table order (TrunkSegment::tile_begin).  CTA b takes the contiguous tile range
// [n_tiles*b/grid, n_tiles*(b+1)/grid) and warp w computes sample w of each tile (trunk_sample).  The CTA stages a
// policy's conv weights only when its next tile belongs to a different policy than the one staged, between two
// __syncthreads(): with the segments of a policy adjacent in the table, a CTA restages at most once per policy
// boundary inside its range.  Warps sync with each other only there.
struct TrunkSegment {
    long long blk_begin;     // env_begin * agents_per_env: the packed block of env 0 of the segment, agent 0
    long long row_begin;     // feature row of sample 0
    long long n_samples;     // n_envs * k
    long long tile_begin;    // first tile of the segment (tiles of all earlier segments before it)
    int policy, k;
    unsigned char ids[CTF_MAX_AGENTS];
};

struct TrunkPolicyWeights {
    const float* conv1_w;
    const float* conv1_b;
    const uint2* conv2_w;
    const float* conv2_b;
};

// The argument block of one launch, passed by value.  Two sizes are instantiated: <1, 1> for a launch with one policy
// and one segment (every ctf_policy_features call), so that the per-pair league path, which is bound by the host,
// does not ship the grouped tables; <CTF_GROUPED_MAX_POLICIES, CTF_GROUPED_MAX_SEGMENTS> for every other launch.
template <int kMaxPolicies, int kMaxSegments>
struct TrunkLaunch {
    TrunkGeometry geo;
    long long n_tiles;
    int n_segments, pad;
    TrunkPolicyWeights w[kMaxPolicies];
    TrunkSegment seg[kMaxSegments];
};
using TrunkLaunchOne = TrunkLaunch<1, 1>;
using TrunkLaunchGrouped = TrunkLaunch<CTF_GROUPED_MAX_POLICIES, CTF_GROUPED_MAX_SEGMENTS>;
static_assert(sizeof(TrunkLaunchOne) <= 256, "a single-policy launch keeps a parameter block of a few hundred bytes");
static_assert(sizeof(TrunkLaunchGrouped) <= 32764, "kernel parameters are limited to 32 764 bytes");

// Both instantiations run one schedule; <1, 1> compiles out the segment search, walk and policy compare and stages its
// one policy's weights before its tiles.  The register cap (5 CTAs of 256 threads per SM) holds both to 48 registers,
// no spills; unbounded they take 126 (grouped) and 111 (<1, 1>), which would cap their residency on small maps.
template <int kMaxPolicies, int kMaxSegments>
__global__ void __launch_bounds__(kTrunkThreads, 5)
k_policy_trunk(const __grid_constant__ TrunkLaunch<kMaxPolicies, kMaxSegments> A) {
    extern __shared__ uint4 smem_raw[];
    const TrunkGeometry& T = A.geo;
    float* w1 = reinterpret_cast<float*>(smem_raw);                      // [C*9][16]: column of one (c, dy, dx) tap
    float* b1 = w1 + T.C * 9 * 16;                                        // [16]
    float* b2 = b1 + 16;                                                  // [32]
    uint2* w2 = reinterpret_cast<uint2*>(b2 + 32);                        // [9][4][32]
    uint32_t* warp_base = reinterpret_cast<uint32_t*>(w2 + kTrunkW2Words / 2);
    const int C = T.C, G = T.G, GG = T.GG, S1 = T.S1, S2 = T.S2, M2 = S2 * S2;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t* bits = warp_base + (size_t)warp * T.warp_words;                           // [wpa]
    uint16_t* cmask = reinterpret_cast<uint16_t*>(bits + T.off_mask);                   // [GG] channel mask per cell
    uint32_t* act = bits + T.off_act;                                                    // [S1*S1][8] bf16x2
    __nv_bfloat16* stage = reinterpret_cast<__nv_bfloat16*>(bits + T.off_stage);        // [8][M2]
    const int g = lane >> 2, t = lane & 3;
    const int n_mt = (M2 + 15) >> 4;
    const long long conv_elems = 32LL * M2;

    const long long t0 = A.n_tiles * blockIdx.x / gridDim.x, t1 = A.n_tiles * (blockIdx.x + 1) / gridDim.x;
    if constexpr (kMaxSegments == 1) {
        // one segment of one policy: its weights are staged once, and the CTA's tiles are its samples in order
        const TrunkSegment& S = A.seg[0];
        const TrunkPolicyWeights& W = A.w[0];
        trunk_stage_weights(W.conv1_w, W.conv1_b, W.conv2_w, W.conv2_b, C, w1, b1, b2, w2);
        __syncthreads();
        const long long s1 = min(t1 * kTrunkWarps, S.n_samples);
        for (long long s = t0 * kTrunkWarps + warp; s < s1; s += kTrunkWarps) {
            const long long e = s / S.k;
            const int j = (int)(s - e * S.k);
            trunk_sample(T, S.blk_begin + e * T.ape + S.ids[j], S.row_begin + s, w1, b1, b2, w2, bits, cmask, act, stage,
                         lane, C, G, GG, S1, S2, M2, g, t, n_mt, conv_elems);
        }
    } else {
        // the segment of tile t0: the last whose first tile is <= t0 (empty segments share their successor's tile_begin)
        int lo = 0, hi = A.n_segments - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (A.seg[mid].tile_begin <= t0) lo = mid; else hi = mid - 1;
        }
        int si = lo, staged = -1;
        for (long long tile = t0; tile < t1; ++tile) {
            while (si + 1 < A.n_segments && A.seg[si + 1].tile_begin <= tile) ++si;
            const TrunkSegment& S = A.seg[si];
            if (S.policy != staged) {
                __syncthreads();
                const TrunkPolicyWeights& W = A.w[S.policy];
                trunk_stage_weights(W.conv1_w, W.conv1_b, W.conv2_w, W.conv2_b, C, w1, b1, b2, w2);
                __syncthreads();
                staged = S.policy;
            }
            const long long s = (tile - S.tile_begin) * kTrunkWarps + warp;
            if (s < S.n_samples) {
                const long long e = s / S.k;
                const int j = (int)(s - e * S.k);
                trunk_sample(T, S.blk_begin + e * T.ape + S.ids[j], S.row_begin + s, w1, b1, b2, w2, bits, cmask, act,
                             stage, lane, C, G, GG, S1, S2, M2, g, t, n_mt, conv_elems);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// backward of the policy trunk: parameter gradients of conv1 / conv2 from packed observations, saved rows and dRows
// ------------------------------------------------------------------------------------------------
// One CTA works on one sample at a time (samples blockIdx.x, + gridDim.x, ...) and accumulates the parameter gradients
// of all its samples in registers; every gradient slot has exactly one owner thread, so there are no atomics.
//   1. stage the packed words; trunk_conv1 rebuilds the channel mask and h1 = bf16(tanh(conv1)) as the forward does;
//      dz2 = bf16(dRow * (1 - h2^2)) (fp32, h2 = the saved row) into a [position][32 channels] tile.
//   2. dW2 (+ db2) on tensor cores: D[co][(tap, ci)] += dz2[co][m] * h1[ci][m + tap], M = 32, K = the (G-4)^2 positions,
//      N = 144 + one column of ones whose product is db2; both operands come from [position][channel] tiles through
//      ldmatrix.trans.  Warp w owns n-tiles w, w + 8, w + 16 of both m-tiles.
//      dh1 = conv2^T(dz2) on tensor cores: M = (G-2)^2 positions, N = 16, K = 9 taps x 32 channels (18 k-steps), B from
//      the transposed fragment layout (fused_policy.conv2_transpose_layout_index); dz1 = dh1 * (1 - h1^2) in fp32.
//   3. dW1 sparsely: thread j owns column (c, tap) = j / 2 and output channels 8 (j & 1) .. + 7 and walks the set bits
//      of channel c, adding dz1 of the output position each one feeds (exact fp32 adds, fixed order); one more column
//      sums dz1 over every position (db1).
// Each CTA writes its partial sums to its row of the workspace; k_policy_grad_reduce sums the rows in index order.
constexpr int kBwdThreads = 256;
constexpr int kBwdWarps = kBwdThreads / 32;
constexpr int kBwdNt = 19;                      // dW2 n-tiles: 18 of (tap, 8 input channels) + the ones column (db2)
constexpr int kBwdW2tWords = 9 * 2 * 2 * 32 * 2;   // conv2^T B fragments: [tap][k-half][n-tile][lane][2 x bf16x2]
// partial sums of one CTA: [dW2 [32][tap*16 + ci] | db2 [32] | dW1 [c*9 + tap][16] | db1 [16]]
constexpr int kGradW2 = 0, kGradB2 = 32 * 144, kGradW1 = kGradB2 + 32;
__host__ __device__ constexpr int grad_count(int C) { return kGradW1 + C * 9 * 16 + 16; }

struct TrunkBwdArgs {
    const float* conv1_w;
    const float* conv1_b;
    const uint2* conv2_wt;
    const uint32_t* packed;
    const __nv_bfloat16* features;
    const __nv_bfloat16* grad_features;
    float* partial;           // [gridDim.x][grad_count(C)]
    long long n_samples;
    long long stride;
    int ape, k;
    int G, C, GG, wpa;
    int S1, S2, K2;           // conv1 / conv2 output side, conv2 positions padded to a multiple of 16
    int off_bits, off_mask, off_act, off_dz2;   // word offsets of the per-sample buffers (dz1 shares the mask's words)
    unsigned char ids[CTF_MAX_AGENTS];
};

__device__ __forceinline__ void ldsm_x4_trans(uint32_t (&r)[4], const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"((unsigned)__cvta_generic_to_shared(p)));
}
__device__ __forceinline__ void ldsm_x2_trans(uint32_t& r0, uint32_t& r1, const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];\n"
                 : "=r"(r0), "=r"(r1) : "r"((unsigned)__cvta_generic_to_shared(p)));
}
__device__ __forceinline__ void mma_bf16(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
// d * (1 - h*h) with one rounding per operation and no contraction, as torch evaluates it in fp32
__device__ __forceinline__ float tanh_grad(float d, float h) { return __fmul_rn(d, __fsub_rn(1.f, __fmul_rn(h, h))); }

// 3 CTAs per SM: 80 registers without spills (126 unbounded = 2 CTAs; 4 CTAs = 64 registers and spills)
__global__ void __launch_bounds__(kBwdThreads, 3) k_policy_trunk_backward(const __grid_constant__ TrunkBwdArgs A) {
    extern __shared__ uint4 smem_raw[];
    float* w1 = reinterpret_cast<float*>(smem_raw);                      // [C*9][16] as in k_policy_trunk
    float* b1 = w1 + A.C * 9 * 16;                                        // [16]
    uint32_t* ones = reinterpret_cast<uint32_t*>(b1 + 16);                // [4]: 8 bf16 ones (one ldmatrix row)
    uint2* w2t = reinterpret_cast<uint2*>(ones + 4);                      // [9][2][2][32]
    uint32_t* base = reinterpret_cast<uint32_t*>(smem_raw);
    uint32_t* bits = base + A.off_bits;                                   // [wpa]
    uint16_t* cmask = reinterpret_cast<uint16_t*>(base + A.off_mask);     // [GG]
    float* dz1 = reinterpret_cast<float*>(base + A.off_mask);            // [S1*S1][16], after conv1 (cmask is dead)
    uint32_t* act = base + A.off_act;                                     // [S1*S1][8] bf16x2 = h1
    __nv_bfloat16* dz2 = reinterpret_cast<__nv_bfloat16*>(base + A.off_dz2);   // [K2][32]
    const uint32_t* dz2w = base + A.off_dz2;
    const int C = A.C, G = A.G, GG = A.GG, S1 = A.S1, S2 = A.S2, M2 = S2 * S2, Q = S1 * S1, K2 = A.K2;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    for (int i = tid; i < C * 9 * 16; i += kBwdThreads) {
        const int o = i & 15, tap = i >> 4;
        w1[i] = A.conv1_w[o * C * 9 + tap];
    }
    if (tid < 16) b1[tid] = A.conv1_b[tid];
    if (tid < 4) ones[tid] = 0x3F803F80u;                                  // bf16 1.0 twice
    for (int i = tid; i < kBwdW2tWords / 2; i += kBwdThreads) w2t[i] = A.conv2_wt[i];

    float accw2[3][2][4];                                                  // [n-tile w + 8i][m-tile][mma D]
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int r = 0; r < 4; ++r) accw2[i][mt][r] = 0.f;
    const int col = tid >> 1, half = tid & 1;                              // dW1 column (c*9 + tap, or C*9: db1)
    const bool has_col = col <= C * 9;
    const int cc = col / 9, ctap = col - cc * 9, cdy = ctap / 3, cdx = ctap - cdy * 3;
    float accw1[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) accw1[o] = 0.f;
    const int n_mt1 = (Q + 15) >> 4;                                        // dh1 m-tiles
    const unsigned div_g = 65536u / (unsigned)G + 1u;                       // p / G = (p * div_g) >> 16 for p < 256

    for (long long s = blockIdx.x; s < A.n_samples; s += gridDim.x) {
        const long long e = s / A.k;
        const int j = (int)(s - e * A.k);
        const long long blk = e * A.ape + A.ids[j];
        const uint32_t* src = A.packed + blk * A.wpa;
        for (int i = tid; i < A.wpa; i += kBwdThreads) bits[i] = __ldg(src + i);
        __syncthreads();                                                   // also orders the weights on the first pass
        trunk_conv1(bits, cmask, act, w1, b1, C, G, GG, S1, tid, kBwdThreads, [] { __syncthreads(); });
        // dz2 = dRow * (1 - h2^2), 8 row elements per 16-byte load; element co*M2 + m goes to dz2[m][co]
        const uint4* hrow = reinterpret_cast<const uint4*>(A.features + s * A.stride);
        const uint4* drow = reinterpret_cast<const uint4*>(A.grad_features + s * A.stride);
        for (int i = tid; i < 4 * M2; i += kBwdThreads) {
            const uint4 hv = __ldg(hrow + i), dv = __ldg(drow + i);
            const __nv_bfloat16* h8 = reinterpret_cast<const __nv_bfloat16*>(&hv);
            const __nv_bfloat16* d8 = reinterpret_cast<const __nv_bfloat16*>(&dv);
            int co = (8 * i) / M2, m = 8 * i - co * M2;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                dz2[m * 32 + co] = __float2bfloat16_rn(tanh_grad(__bfloat162float(d8[u]), __bfloat162float(h8[u])));
                if (++m == M2) { m = 0; ++co; }
            }
        }
        for (int i = M2 * 16 + tid; i < K2 * 16; i += kBwdThreads) base[A.off_dz2 + i] = 0u;   // K padding rows
        __syncthreads();

        // dW2 and db2: A = dz2 (rows co), B = h1 at position m + tap (columns (tap, ci)) or ones
        for (int k0 = 0; k0 < K2; k0 += 16) {
            uint32_t a[2][4];
            {
                const int mat = lane >> 3, m = k0 + (mat >> 1) * 8 + (lane & 7);
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) ldsm_x4_trans(a[mt], dz2 + m * 32 + 16 * mt + (mat & 1) * 8);
            }
            const int mb = min(k0 + (lane & 15), M2 - 1);                   // pad rows: A is zero there
            const int yb = mb / S2, pb = yb * S1 + (mb - yb * S2);
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const int nt = warp + 8 * i;
                if (nt < kBwdNt) {
                    const int tap = nt >> 1;
                    const void* bp = nt == 18 ? static_cast<const void*>(ones)
                                              : static_cast<const void*>(act + (pb + (tap / 3) * S1 + tap % 3) * 8 + (nt & 1) * 4);
                    uint32_t b0, b1r;
                    ldsm_x2_trans(b0, b1r, bp);
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt) mma_bf16(accw2[i][mt], a[mt][0], a[mt][1], a[mt][2], a[mt][3], b0, b1r);
                }
            }
        }
        // dh1 = conv2^T(dz2) per (m-tile of conv1 positions, n-tile of 8 input channels); dz1 = dh1 * (1 - h1^2)
        for (int job = (warp + 5) & 7; job < 2 * n_mt1; job += kBwdWarps) {
            const int mt = job >> 1, nt = job & 1;
            const int q0 = mt * 16 + g, q1 = q0 + 8;
            const int y0 = q0 / S1, x0 = q0 - y0 * S1, y1 = q1 / S1, x1 = q1 - y1 * S1;
            float d[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
                const int dy = tap / 3, dx = tap % 3;
                const int r0y = y0 - dy, r0x = x0 - dx, r1y = y1 - dy, r1x = x1 - dx;
                const bool v0 = q0 < Q && (unsigned)r0y < (unsigned)S2 && (unsigned)r0x < (unsigned)S2;
                const bool v1 = q1 < Q && (unsigned)r1y < (unsigned)S2 && (unsigned)r1x < (unsigned)S2;
                const int m0 = v0 ? r0y * S2 + r0x : 0, m1 = v1 ? r1y * S2 + r1x : 0;
#pragma unroll
                for (int kh = 0; kh < 2; ++kh) {
                    const uint32_t a0 = v0 ? dz2w[m0 * 16 + kh * 8 + t] : 0u, a2 = v0 ? dz2w[m0 * 16 + kh * 8 + 4 + t] : 0u;
                    const uint32_t a1 = v1 ? dz2w[m1 * 16 + kh * 8 + t] : 0u, a3 = v1 ? dz2w[m1 * 16 + kh * 8 + 4 + t] : 0u;
                    const uint2 b = w2t[((tap * 2 + kh) * 2 + nt) * 32 + lane];
                    mma_bf16(d, a0, a1, a2, a3, b.x, b.y);
                }
            }
            const int ci = nt * 8 + 2 * t;
            if (q0 < Q) {
                const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(act + q0 * 8 + (ci >> 1));
                *reinterpret_cast<float2*>(dz1 + q0 * 16 + ci) =
                    make_float2(tanh_grad(d[0], __low2float(h)), tanh_grad(d[1], __high2float(h)));
            }
            if (q1 < Q) {
                const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(act + q1 * 8 + (ci >> 1));
                *reinterpret_cast<float2*>(dz1 + q1 * 16 + ci) =
                    make_float2(tanh_grad(d[2], __low2float(h)), tanh_grad(d[3], __high2float(h)));
            }
        }
        __syncthreads();

        // dW1: the set bits of channel cc feed output position (cell - tap) when it is inside the conv1 output
        if (has_col) {
            const float4* z = reinterpret_cast<const float4*>(dz1) + half * 2;
            if (col < C * 9) {
                const int el0 = cc * GG, el1 = el0 + GG;
                for (int w = el0 >> 5; w <= (el1 - 1) >> 5; ++w) {
                    uint32_t m = bits[w];
                    if (32 * w < el0) m &= ~0u << (el0 - 32 * w);
                    if (32 * w + 32 > el1) m &= ~0u >> (32 * w + 32 - el1);
                    while (m) {
                        const int p = 32 * w + __ffs(m) - 1 - el0;
                        m &= m - 1;
                        const int py = (int)(((unsigned)p * div_g) >> 16), px = p - py * G;
                        const int qy = py - cdy, qx = px - cdx;
                        if ((unsigned)qy < (unsigned)S1 && (unsigned)qx < (unsigned)S1) {
                            const float4 u = z[(qy * S1 + qx) * 4], v = z[(qy * S1 + qx) * 4 + 1];
                            accw1[0] += u.x; accw1[1] += u.y; accw1[2] += u.z; accw1[3] += u.w;
                            accw1[4] += v.x; accw1[5] += v.y; accw1[6] += v.z; accw1[7] += v.w;
                        }
                    }
                }
            } else {
                for (int q = 0; q < Q; ++q) {
                    const float4 u = z[q * 4], v = z[q * 4 + 1];
                    accw1[0] += u.x; accw1[1] += u.y; accw1[2] += u.z; accw1[3] += u.w;
                    accw1[4] += v.x; accw1[5] += v.y; accw1[6] += v.z; accw1[7] += v.w;
                }
            }
        }
        __syncthreads();
    }

    // partial sums of this CTA (zeros when it had no sample)
    float* out = A.partial + (size_t)blockIdx.x * grad_count(C);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const int nt = warp + 8 * i;
        if (nt < kBwdNt) {
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                const int co = mt * 16 + g;
                if (nt < 18) {
                    const int n = nt * 8 + 2 * t;
                    *reinterpret_cast<float2*>(out + kGradW2 + co * 144 + n) = make_float2(accw2[i][mt][0], accw2[i][mt][1]);
                    *reinterpret_cast<float2*>(out + kGradW2 + (co + 8) * 144 + n) = make_float2(accw2[i][mt][2], accw2[i][mt][3]);
                } else if (t == 0) {                                                         // column 0 of the ones tile
                    out[kGradB2 + co] = accw2[i][mt][0];
                    out[kGradB2 + co + 8] = accw2[i][mt][2];
                }
            }
        }
    }
    if (has_col) {
        float4* o = reinterpret_cast<float4*>(out + kGradW1 + col * 16 + half * 8);
        o[0] = make_float4(accw1[0], accw1[1], accw1[2], accw1[3]);
        o[1] = make_float4(accw1[4], accw1[5], accw1[6], accw1[7]);
    }
}

// Sums the n_parts partial rows in row order (fixed, so reruns are bit-identical) and writes the gradients in torch
// layout: thread i produces element i of [conv1.weight [16][C][3][3] | conv1.bias | conv2.weight [32][16][3][3] | conv2.bias].
__global__ void k_policy_grad_reduce(const float* __restrict__ partial, int n_parts, int C, float* __restrict__ g_c1w,
                                     float* __restrict__ g_c1b, float* __restrict__ g_c2w, float* __restrict__ g_c2b) {
    const int n_c1w = 16 * C * 9, n = grad_count(C);
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int src;
    float* dst;
    if (i < n_c1w) {
        const int o = i / (C * 9), col = i - o * C * 9;                  // col = c*9 + tap
        src = kGradW1 + col * 16 + o; dst = g_c1w + i;
    } else if ((i -= n_c1w) < 16) {
        src = kGradW1 + C * 9 * 16 + i; dst = g_c1b + i;
    } else if ((i -= 16) < 32 * 144) {
        const int co = i / 144, r = i - co * 144, ci = r / 9, tap = r - ci * 9;
        src = kGradW2 + co * 144 + tap * 16 + ci; dst = g_c2w + i;
    } else if ((i -= 32 * 144) < 32) {
        src = kGradB2 + i; dst = g_c2b + i;
    } else {
        return;
    }
    float acc = 0.f;
#pragma unroll 8
    for (int p = 0; p < n_parts; ++p) acc += __ldg(partial + (size_t)p * n + src);
    *dst = acc;
}

// shared-memory layout of k_policy_trunk_backward for a plan
static __host__ void trunk_bwd_layout(const DevPlan& P, TrunkBwdArgs& A, size_t& smem) {
    const int S1 = P.G - 2, S2 = P.G - 4;
    const auto up4 = [](int w) { return (w + 3) & ~3; };
    A.G = P.G; A.C = P.C; A.GG = P.GG; A.wpa = P.wpa; A.S1 = S1; A.S2 = S2; A.K2 = (S2 * S2 + 15) & ~15;
    A.off_bits = P.C * 9 * 16 + 16 + 4 + kBwdW2tWords;                 // after w1, b1, ones, w2t (all 16-byte multiples)
    A.off_mask = A.off_bits + up4(P.wpa);
    const int mask_words = up4((P.GG + 1) / 2), dz1_words = S1 * S1 * 16;
    A.off_act = A.off_mask + (mask_words > dz1_words ? mask_words : dz1_words);
    A.off_dz2 = A.off_act + S1 * S1 * 8;
    smem = (size_t)(A.off_dz2 + A.K2 * 16) * 4;
}

// ================================================================================================
// k_gae — generalised advantage estimation over a rollout, one thread per (trained agent, env) column
// ================================================================================================
constexpr int kGaeThreads = 256;
constexpr int kGaeUnroll = 8;   // rows whose loads are issued before the recurrence consumes the first of them
// 6 CTAs per SM leave 40 registers, enough for the 16 loads in flight without spills (8 CTAs spill); the 24 loads of
// k_gae<true> spill at 40 registers, so it runs 5 CTAs per SM (48 registers)

// Rows are [T*apt][B] fp32 with row t*apt + j = agent j at step t, so column c = j*B + b of a row is contiguous over
// the threads of a warp: every load and store is coalesced.  The recurrence runs backwards over t with one explicit
// rounding per operation (no FMA contraction), which is bit for bit the eager torch statement ppo.reference_advantages:
//   delta = (r[t] + gamma*nv) - v[t];  last = delta + gamma_lambda*last;  adv[t] = last;  ret[t] = last + v[t]
// with nv = next_value for t = T-1 and v[t+1] below it.
// kDones (ctf_gae_dones): a nonzero dones[t] means observation t starts a new episode (CleanRL's convention), so after
// row t both nv and last are selected to exactly 0 before row t-1: no bootstrap and no advantage crosses the boundary.
// dones is the last parameter so that the other parameters keep their offsets and k_gae<false> its code.
template <bool kDones>
__global__ void __launch_bounds__(kGaeThreads, kDones ? 5 : 6) k_gae(const float* __restrict__ rewards, const float* __restrict__ values,
                                                     const float* __restrict__ next_value, float* __restrict__ adv,
                                                     float* __restrict__ ret, long long T, long long cols, float gamma,
                                                     float gamma_lambda, const float* __restrict__ dones) {
    const long long c = (long long)blockIdx.x * kGaeThreads + threadIdx.x;
    if (c >= cols) return;
    float nv = __ldg(next_value + c), last = 0.f;
    long long t = T - 1;
    for (; t >= kGaeUnroll - 1; t -= kGaeUnroll) {
        float r[kGaeUnroll], v[kGaeUnroll], d[kGaeUnroll];
#pragma unroll
        for (int u = 0; u < kGaeUnroll; ++u) {
            const size_t i = (size_t)(t - u) * cols + c;
            r[u] = __ldcs(rewards + i);
            v[u] = __ldcs(values + i);
            if (kDones) d[u] = __ldcs(dones + i);
        }
#pragma unroll
        for (int u = 0; u < kGaeUnroll; ++u) {
            const size_t i = (size_t)(t - u) * cols + c;
            const float delta = __fsub_rn(__fadd_rn(r[u], __fmul_rn(gamma, nv)), v[u]);
            last = __fadd_rn(delta, __fmul_rn(gamma_lambda, last));
            __stcs(adv + i, last);
            __stcs(ret + i, __fadd_rn(last, v[u]));
            nv = v[u];
            if (kDones && d[u] != 0.f) nv = last = 0.f;
        }
    }
    for (; t >= 0; --t) {
        const size_t i = (size_t)t * cols + c;
        const float r = __ldcs(rewards + i), v = __ldcs(values + i);
        const bool start = kDones && __ldcs(dones + i) != 0.f;
        const float delta = __fsub_rn(__fadd_rn(r, __fmul_rn(gamma, nv)), v);
        last = __fadd_rn(delta, __fmul_rn(gamma_lambda, last));
        __stcs(adv + i, last);
        __stcs(ret + i, __fadd_rn(last, v));
        nv = v;
        if (start) nv = last = 0.f;
    }
}

// ================================================================================================
// k_sample_actions — one seeded categorical draw per policy row (ctf_sample_actions), one thread per row
// ================================================================================================
constexpr int kSampleThreads = 256;
constexpr uint32_t kPolicySite = 0x80000000u;   // top bit of the counter's site word: disjoint from the env's sites 0..31
constexpr int kNoOpAction = 4;

// Row r is agent a = flat_index[r] % N of env b = flat_index[r] / N.  Its draw is word 0 of Philox4x32-10 at counter
// (env_id_base + b, episode[b], step_count[b], kPolicySite | a), read from the env state at launch, so the result of a
// row depends on nothing but its logits, its mask flag and (seed, global env id, episode, step, agent).  Every add and
// multiply is rounded on its own, so the action does not depend on the compiler contracting anything into an FMA
// (marl_ctf_development_b200/draws.py: sample_action states it in float64).  The action is in 0..8 whatever the logits:
// with no positive mass at all (NaN or infinite logits) it is the no-op 4.  A flat_index outside [0, B*N) writes
// nothing and sets CTF_FAULT_BAD_INDEX, the only atomic (an idempotent OR into the fault word, as k_step reports its
// faults): the outputs themselves are plain stores, bit-identical from run to run.
__global__ void __launch_bounds__(kSampleThreads) k_sample_actions(
    const float* __restrict__ head, long long head_stride, const uint8_t* __restrict__ masked,
    const long long* __restrict__ flat_index, long long n_rows, const uint4* __restrict__ envs, long long n_flat,
    int n_agents, uint32_t env_id_base, uint32_t seed_lo, uint32_t seed_hi, uint8_t* __restrict__ actions,
    long long* __restrict__ action_out, float* __restrict__ logprob, float* __restrict__ entropy,
    uint32_t* __restrict__ faults) {
    const long long r = (long long)blockIdx.x * kSampleThreads + threadIdx.x;
    if (r >= n_rows) return;
    const long long f = __ldg(flat_index + r);
    if (f < 0 || f >= n_flat) {
        atomicOr(faults, CTF_FAULT_BAD_INDEX);
        return;
    }
    const long long b = f / n_agents;
    const uint32_t a = (uint32_t)(f - b * n_agents);
    const uint4 ev = envs[b];   // x = env_step_count, y = episode
    uint32_t w[4];
    philox4x32_10(env_id_base + (uint32_t)b, ev.y, ev.x, kPolicySite | a, seed_lo, seed_hi, w);
    const float u = __fmul_rn((float)(w[0] >> 8), 0x1p-24f);

    const float* row = head + r * head_stride + 1;
    const bool mask = masked != nullptr && __ldg(masked + r) != 0;
    float x[CTF_N_ACTIONS];
    float m = -INFINITY;
#pragma unroll
    for (int i = 0; i < CTF_N_ACTIONS; ++i) {
        x[i] = __ldg(row + i);
        if (mask && i >= 5) x[i] = __fadd_rn(x[i], -1e9f);   // CtfPolicy.masked_logits
        m = fmaxf(m, x[i]);
    }
    float e[CTF_N_ACTIONS], z = 0.f;
#pragma unroll
    for (int i = 0; i < CTF_N_ACTIONS; ++i) {
        e[i] = expf(__fsub_rn(x[i], m));
        z = __fadd_rn(z, e[i]);
    }
    const float t = __fmul_rn(u, z);
    int act = -1, last_pos = kNoOpAction;
    float c = 0.f, s = 0.f;
#pragma unroll
    for (int i = 0; i < CTF_N_ACTIONS; ++i) {
        c = __fadd_rn(c, e[i]);
        if (act < 0 && t < c) act = i;
        if (e[i] > 0.f) {
            last_pos = i;
            s = __fadd_rn(s, __fmul_rn(e[i], __fsub_rn(x[i], m)));
        }
    }
    if (act < 0) act = last_pos;
    float x_act = x[0];
#pragma unroll
    for (int i = 1; i < CTF_N_ACTIONS; ++i) x_act = i == act ? x[i] : x_act;   // a select: x stays in registers
    const float log_z = logf(z);
    if (actions) actions[f] = (uint8_t)act;
    if (action_out) action_out[r] = act;
    if (logprob) logprob[r] = __fsub_rn(__fsub_rn(x_act, m), log_z);
    if (entropy) entropy[r] = __fsub_rn(log_z, __fdiv_rn(s, z));
}

}  // namespace

// ================================================================================================
// Host side: C ABI
// ================================================================================================
struct ctf_env {
    DevPlan plan;
    ctf_config_t cfg;
    long long B;
    int device;
    int stats_level;
    int obs_dtype;
    uint64_t seed;
    uint64_t env_id_base;
    uint32_t* faults;        // device
    uint8_t* actions_stage;  // device [B][N], for ctf_step_host
    float* rewards_stage;    // device [B][N], used by ctf_step_host when out.rewards is NULL
    uint8_t* dones_stage;    // device [B]
    size_t smem_bytes;       // warp-per-env kernels writing a plain observation buffer (padded to the residency cap)
    size_t smem_bytes_comp;  // the same kernels writing a compressed one (a different cap, see ctf_create)
    size_t smem_bytes_delta; // k_step writing the buffer that has a record (delta writes, logic-bound)
    const void* obs_seen;    // the last outputs.obs launched on, and whether it lies in compressed memory
    bool obs_seen_comp;
    const void* rec_obs;     // ctf_bind_obs_record: the buffer whose record is kept, and the record (device)
    uint32_t* record;
    uint32_t* record_epoch;
    const uint32_t* epoch;
    size_t trunk_smem_bytes; // k_policy_trunk: dynamic shared memory for this plan
    int trunk_ctas;          // k_policy_trunk<1, 1>: CTAs that fit on the device at once
    int grouped_ctas;        // k_policy_trunk<CTF_GROUPED_MAX_POLICIES, CTF_GROUPED_MAX_SEGMENTS>: the same
    size_t bwd_smem_bytes;   // k_policy_trunk_backward: dynamic shared memory for this plan
    int bwd_ctas;            // k_policy_trunk_backward: CTAs (= workspace rows) of every launch with >= bwd_ctas samples
};

// cudaSetDevice for the duration of an entry point; the caller's current device is restored on return
struct DeviceGuard {
    int prev = -1;
    cudaError_t err;
    explicit DeviceGuard(int device) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != device) err = cudaSetDevice(device);
        else if (err == cudaSuccess) prev = -1;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, const char* a = "", const char* b = "") {
    snprintf(g_err, sizeof(g_err), fmt, a, b);
    return code;
}

#define CTF_CUDA(call)                                                              \
    do {                                                                            \
        cudaError_t e_ = (call);                                                    \
        if (e_ != cudaSuccess) return fail(CTF_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

extern "C" const char* ctf_last_error(void) { return g_err; }
extern "C" int ctf_abi_version(void) { return CTF_ABI_VERSION; }
extern "C" size_t ctf_config_size(void) { return sizeof(ctf_config_t); }

// ------------------------------------------------------------------ compressible device memory (DESIGN §4)
// The driver's virtual-memory entry points, resolved through the runtime so that the library does not link libcuda.
struct VmmApi {
    PFN_cuGetErrorString err_str = nullptr;
    PFN_cuDeviceGetAttribute dev_attr = nullptr;
    PFN_cuMemGetAllocationGranularity granularity = nullptr;
    PFN_cuMemCreate create = nullptr;
    PFN_cuMemRelease release = nullptr;
    PFN_cuMemAddressReserve reserve = nullptr;
    PFN_cuMemAddressFree addr_free = nullptr;
    PFN_cuMemMap map = nullptr;
    PFN_cuMemUnmap unmap = nullptr;
    PFN_cuMemSetAccess set_access = nullptr;
    PFN_cuMemRetainAllocationHandle retain = nullptr;
    PFN_cuMemGetAllocationPropertiesFromHandle props = nullptr;
    const char* missing = nullptr;   // the first entry point the driver did not provide
};

static const VmmApi& vmm_api() {
    static VmmApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        auto get = [](const char* sym, auto& fn) {
            void* p = nullptr;
            cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
            if (cudaGetDriverEntryPointByVersion(sym, &p, 12000, cudaEnableDefault, &q) != cudaSuccess ||
                q != cudaDriverEntryPointSuccess || !p) {
                if (!api.missing) api.missing = sym;
                return;
            }
            fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(p);
        };
        get("cuGetErrorString", api.err_str);
        get("cuDeviceGetAttribute", api.dev_attr);
        get("cuMemGetAllocationGranularity", api.granularity);
        get("cuMemCreate", api.create);
        get("cuMemRelease", api.release);
        get("cuMemAddressReserve", api.reserve);
        get("cuMemAddressFree", api.addr_free);
        get("cuMemMap", api.map);
        get("cuMemUnmap", api.unmap);
        get("cuMemSetAccess", api.set_access);
        get("cuMemRetainAllocationHandle", api.retain);
        get("cuMemGetAllocationPropertiesFromHandle", api.props);
    });
    return api;
}

static int cu_fail(const VmmApi& api, const char* what, CUresult r) {
    const char* msg = nullptr;
    if (api.err_str) api.err_str(r, &msg);
    return fail(CTF_ERR_CUDA, "%s: %s", what, msg ? msg : "unknown CUDA driver error");
}

struct VmmBlock {
    CUmemGenericAllocationHandle handle;
    size_t bytes;   // mapped size (the request rounded up to the granularity)
};
// never destroyed: torch may free its cached blocks after this library's static destructors have run
static std::mutex* const g_vmm_mu = new std::mutex;
static std::unordered_map<uintptr_t, VmmBlock>* const g_vmm_blocks = new std::unordered_map<uintptr_t, VmmBlock>;
static std::atomic<int> g_compression_enabled{1};

static int compression_supported(const VmmApi& api, int device, int* out) {
    if (api.missing) return fail(CTF_ERR_CUDA, "the CUDA driver does not provide %s", api.missing);
    int v = 0;
    CUresult r = api.dev_attr(&v, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, (CUdevice)device);
    if (r != CUDA_SUCCESS) return cu_fail(api, "cuDeviceGetAttribute(GENERIC_COMPRESSION_SUPPORTED)", r);
    *out = v ? 1 : 0;
    return CTF_OK;
}

static int vmm_alloc(int device, size_t size, void** out) {
    const VmmApi& api = vmm_api();
    DeviceGuard guard(device);   // the runtime's primary context is current for the driver calls
    CTF_CUDA(guard.err);
    int supported = 0;
    int rc = compression_supported(api, device, &supported);
    if (rc != CTF_OK) return rc;
    CUmemAllocationProp prop;
    memset(&prop, 0, sizeof(prop));
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = device;
    prop.allocFlags.compressionType =
        supported && g_compression_enabled.load() ? CU_MEM_ALLOCATION_COMP_GENERIC : CU_MEM_ALLOCATION_COMP_NONE;
    CUmemGenericAllocationHandle handle;
    size_t gran = 0, bytes = 0;
    for (;;) {
        CUresult r = api.granularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED);
        if (r != CUDA_SUCCESS) return cu_fail(api, "cuMemGetAllocationGranularity", r);
        bytes = ((size > 0 ? size : 1) + gran - 1) / gran * gran;
        r = api.create(&handle, bytes, &prop, 0);
        if (r == CUDA_SUCCESS) break;
        if (prop.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_NONE) return cu_fail(api, "cuMemCreate", r);
        prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_NONE;   // compression refused: ordinary memory instead
    }
    CUdeviceptr ptr = 0;
    CUresult r = api.reserve(&ptr, bytes, gran, 0, 0);
    if (r != CUDA_SUCCESS) { api.release(handle); return cu_fail(api, "cuMemAddressReserve", r); }
    r = api.map(ptr, bytes, 0, handle, 0);
    if (r != CUDA_SUCCESS) { api.addr_free(ptr, bytes); api.release(handle); return cu_fail(api, "cuMemMap", r); }
    CUmemAccessDesc access;
    memset(&access, 0, sizeof(access));
    access.location = prop.location;
    access.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    r = api.set_access(ptr, bytes, &access, 1);
    if (r != CUDA_SUCCESS) {
        api.unmap(ptr, bytes); api.release(handle); api.addr_free(ptr, bytes);
        return cu_fail(api, "cuMemSetAccess", r);
    }
    {
        std::lock_guard<std::mutex> lock(*g_vmm_mu);
        (*g_vmm_blocks)[(uintptr_t)ptr] = VmmBlock{handle, bytes};
    }
    *out = reinterpret_cast<void*>(ptr);
    return CTF_OK;
}

extern "C" void* ctf_compressible_alloc(ssize_t size, int device, void* /*stream*/) {
    if (size < 0) { fail(CTF_ERR_INVALID, "ctf_compressible_alloc: negative size"); return nullptr; }
    void* p = nullptr;
    return vmm_alloc(device, (size_t)size, &p) == CTF_OK ? p : nullptr;
}

extern "C" void ctf_compressible_free(void* p, ssize_t /*size*/, int device, void* /*stream*/) {
    if (!p) return;
    VmmBlock b;
    {
        std::lock_guard<std::mutex> lock(*g_vmm_mu);
        auto it = g_vmm_blocks->find((uintptr_t)p);
        if (it == g_vmm_blocks->end()) { fail(CTF_ERR_INVALID, "ctf_compressible_free: not a ctf_compressible_alloc pointer"); return; }
        b = it->second;
        g_vmm_blocks->erase(it);
    }
    const VmmApi& api = vmm_api();
    DeviceGuard guard(device);
    const CUdeviceptr ptr = (CUdeviceptr)(uintptr_t)p;
    api.unmap(ptr, b.bytes);
    api.release(b.handle);
    api.addr_free(ptr, b.bytes);
}

extern "C" int ctf_compression_supported(int device, int* out) {
    if (!out) return fail(CTF_ERR_INVALID, "null argument");
    *out = 0;
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) return fail(CTF_ERR_NO_DEVICE, "no CUDA device");
    if (device < 0 || device >= n_dev) return fail(CTF_ERR_INVALID, "device index out of range");
    return compression_supported(vmm_api(), device, out);
}

extern "C" int ctf_mem_is_compressed(const void* p, int* out) {
    if (!out) return fail(CTF_ERR_INVALID, "null argument");
    *out = 0;
    if (!p) return CTF_OK;
    const VmmApi& api = vmm_api();
    if (api.missing) return fail(CTF_ERR_CUDA, "the CUDA driver does not provide %s", api.missing);
    CUmemGenericAllocationHandle h;
    if (api.retain(&h, const_cast<void*>(p)) != CUDA_SUCCESS) return CTF_OK;   // not in a cuMemMap'ed range
    CUmemAllocationProp prop;
    memset(&prop, 0, sizeof(prop));
    CUresult r = api.props(&prop, h);
    api.release(h);   // the reference cuMemRetainAllocationHandle took
    if (r != CUDA_SUCCESS) return cu_fail(api, "cuMemGetAllocationPropertiesFromHandle", r);
    *out = prop.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC ? 1 : 0;
    return CTF_OK;
}

extern "C" int ctf_compressible_set_enabled(int enabled) { return g_compression_enabled.exchange(enabled ? 1 : 0); }

static int build_plan(const ctf_config_t& c, int stats_level, int obs_dtype, DevPlan& P) {
    memset(&P, 0, sizeof(P));
    if (c.grid_size < 2 || c.grid_size > CTF_MAX_GRID) return fail(CTF_ERR_INVALID, "grid_size out of range");
    if (c.n_agents < 1 || c.n_agents > CTF_MAX_AGENTS) return fail(CTF_ERR_INVALID, "n_agents out of range");
    if (c.n_channels < 1 || c.n_channels > CTF_MAX_CHANNELS) return fail(CTF_ERR_INVALID, "n_channels out of range");
    if (c.flip_axis < -1 || c.flip_axis > 2) return fail(CTF_ERR_INVALID, "flip_axis must be -1, 0, 1 or 2");
    if (c.game_steps < 1) return fail(CTF_ERR_INVALID, "game_steps must be positive");
    if (obs_dtype < CTF_OBS_F32 || obs_dtype > CTF_OBS_BF16) return fail(CTF_ERR_INVALID, "unknown obs dtype");
    const int G = c.grid_size, N = c.n_agents;
    P.tag_threshold = c.tag_threshold;
    P.reward_step = c.reward_step; P.reward_capture = c.reward_capture; P.reward_tag = c.reward_tag;
    P.capture_punish = c.capture_punish; P.win_margin = c.win_margin_scalar; P.loss_margin = c.loss_margin_scalar;
    P.G = G; P.N = N; P.C = c.n_channels; P.GG = G * G; P.M = 6 + 2 * N; P.E = N * c.n_channels * G * G;
    P.bits_words = (((P.E + 128 + 31) / 32 + 1) + 15) / 16 * 16;  // pad (<= 127 bits) + 1 slack word, whole 16-word groups
    P.wpa = (c.n_channels * G * G + 31) / 32;
    P.game_steps = c.game_steps; P.flip_axis = c.flip_axis;
    {   // out[i][j] = in[fr][fc] with (fr, fc) = (G1-r, G1-c) both axes, (G1-r, c) rows, (r, G1-c) columns, (G1-c, G1-r) anti-diagonal
        const int G1 = G - 1;
        switch (c.flip_axis) {
            case -1: P.flip_a = -G; P.flip_b = -1; P.flip_d = G1 * G + G1; break;
            case 0: P.flip_a = -G; P.flip_b = 1; P.flip_d = G1 * G; break;
            case 1: P.flip_a = G; P.flip_b = -1; P.flip_d = G1; break;
            default: P.flip_a = -1; P.flip_b = -G; P.flip_d = G1 * G + G1; break;
        }
    }
    P.use_adjusted_rewards = c.use_adjusted_rewards; P.home_flag_capture = c.home_flag_capture;
    P.drop_flag_when_no_hp = c.drop_flag_when_no_hp; P.reverse_team1_actions = c.reverse_team1_actions;
    P.heal_q = c.heal_q; P.vault_cost_q = c.vault_cost_q; P.vault_min_q = c.vault_min_q;
    P.zone_distance = c.zone_distance; P.guardian_distance = c.guardian_distance; P.tagging_range = c.tagging_range;
    P.max_agent_blocks = c.max_agent_blocks; P.block_pickup_value = c.block_pickup_value;
    P.hp_float = c.hp_float ? 1 : 0;
    P.heal_f = c.heal_f; P.vault_cost_f = c.vault_cost_f; P.vault_min_f = c.vault_min_f;
    for (int t = 0; t < 4; ++t) {
        if (P.hp_float) {
            if (!(c.hp_max_f[t] > 0.0)) return fail(CTF_ERR_INVALID, "hp_max_f must be positive");
        } else if (c.hp_max_q[t] <= 0 || c.hp_max_q[t] > 32000) {
            return fail(CTF_ERR_INVALID, "hp_max_q out of int16 range");
        }
        P.hp_max_q[t] = P.hp_float ? 1 : c.hp_max_q[t]; P.damage_q[t] = c.damage_q[t]; P.damage_boosted_q[t] = c.damage_boosted_q[t];
        P.hp_max_f[t] = c.hp_max_f[t]; P.damage_f[t] = c.damage_f[t]; P.damage_boosted_f[t] = c.damage_boosted_f[t];
    }
    for (int i = 0; i < N; ++i) {
        if (c.agent_team[i] > 1 || c.agent_type[i] > 3) return fail(CTF_ERR_INVALID, "agent team/type out of range");
        if (c.start_row[i] >= G || c.start_col[i] >= G) return fail(CTF_ERR_INVALID, "agent start outside the grid");
        if (c.meta_hp_src[i] >= N) return fail(CTF_ERR_INVALID, "meta_hp_src outside 0..N-1");
        P.team[i] = c.agent_team[i]; P.type[i] = c.agent_type[i]; P.tile[i] = c.agent_tile[i];
        P.start_r[i] = c.start_row[i]; P.start_c[i] = c.start_col[i];
        P.obs_rev[i] = c.obs_reverse[i]; P.meta_hp_src[i] = c.meta_hp_src[i];
        P.my_slot[i] = -1;
    }
    for (int t = 0; t < 2; ++t) {
        if (c.n_opponents[t] > 4) return fail(CTF_ERR_INVALID, "more than 4 opponents per team");
        P.n_opp[t] = c.n_opponents[t];
        for (int j = 0; j < c.n_opponents[t]; ++j) {
            const int k = c.opponents[t][j];
            if (k >= N || c.agent_team[k] != 1 - t) return fail(CTF_ERR_INVALID, "opponents list inconsistent with teams");
            if (j > 0 && c.opponents[t][j - 1] >= k) return fail(CTF_ERR_INVALID, "opponents list must be in id order");
            P.my_slot[k] = (signed char)j;
        }
        for (int d = 0; d < 2; ++d) {
            if (c.flag_pos[t][d] >= G || c.capture_pos[t][d] >= G || c.spawn_pos[t][d] >= G)
                return fail(CTF_ERR_INVALID, "flag/capture/spawn position outside the grid");
            if (c.spawn_pos[t][d] < 1) return fail(CTF_ERR_INVALID, "spawn positions need row, col >= 1");
            P.flag_pos[t][d] = c.flag_pos[t][d]; P.capture_pos[t][d] = c.capture_pos[t][d]; P.spawn_pos[t][d] = c.spawn_pos[t][d];
        }
        P.flag_tile[t] = c.flag_tile[t];
        unsigned long long lut = 0;
        for (int tile = 0; tile < CTF_N_TILE_CODES; ++tile) {
            if (c.chan_lut[t][tile] >= c.n_channels) return fail(CTF_ERR_INVALID, "chan_lut entry >= n_channels");
            lut |= (unsigned long long)(c.chan_lut[t][tile] & 15) << (4 * tile);
        }
        P.lut64[t] = lut;
    }
    for (int t = 0; t < 4; ++t)
        for (int a = 0; a < CTF_N_ACTIONS; ++a) { P.delta[t][a][0] = c.action_delta[t][a][0]; P.delta[t][a][1] = c.action_delta[t][a][1]; }
    for (int a = 0; a < 16; ++a) P.rev_action[a] = a < CTF_N_ACTIONS ? c.reversed_action[a] : 4;
    for (int a = 0; a < CTF_N_ACTIONS; ++a)
        if (c.reversed_action[a] >= CTF_N_ACTIONS) return fail(CTF_ERR_INVALID, "reversed_action out of range");
    // metadata slot order (:1050-1067): self, team-mates in id order without self, opponents in id order
    for (int a = 0; a < N; ++a) {
        int q = 0;
        unsigned int row = 0xFFFFFFFFu;
        auto put = [&](int agent) { row = (row & ~(0xFu << (4 * q))) | ((unsigned)agent << (4 * q)); ++q; };
        put(a);
        const int team = c.agent_team[a];
        for (int j = 0; j < c.n_opponents[1 - team]; ++j)
            if (c.opponents[1 - team][j] != a && q < N) put(c.opponents[1 - team][j]);
        for (int j = 0; j < c.n_opponents[team]; ++j)
            if (q < N) put(c.opponents[team][j]);
        P.meta_row[a] = row;
    }
    // the same layout as one code per element (write_meta's float4 path)
    {
        unsigned char codes[256];
        memset(codes, kMetaZero, sizeof(codes));
        const int M = 6 + 2 * N;
        for (int a = 0; a < N; ++a) {
            unsigned char* row = codes + a * M;
            row[0] = kMetaPct;
            row[1] = c.agent_team[a] == 0 ? kMetaRatio0 : kMetaRatio1;
            for (int t = 0; t < 4; ++t) row[2 + t] = (t == c.agent_type[a]) ? kMetaOne : kMetaZero;
            for (int q = 0; q < N; ++q) {
                const unsigned srcAgent = (P.meta_row[a] >> (4 * q)) & 15u;
                row[6 + 2 * q] = srcAgent == 15u ? kMetaZero : (unsigned char)(kMetaHp + srcAgent);
                row[7 + 2 * q] = srcAgent == 15u ? kMetaZero : (unsigned char)(kMetaFlag + srcAgent);
            }
        }
        for (int k = 0; k < 64; ++k)
            P.meta_codes[k] = codes[4 * k] | (codes[4 * k + 1] << 8) | (codes[4 * k + 2] << 16) | ((unsigned)codes[4 * k + 3] << 24);
    }
    for (int r = 0; r < G; ++r)
        for (int cc = 0; cc < G; ++cc) {
            const uint8_t t = c.grid_template[r * G + cc];
            if (t >= CTF_N_TILE_CODES) return fail(CTF_ERR_INVALID, "grid_template holds an unknown tile code");
            P.grid_template[r * kRow + cc] = t;
        }
    // shared-memory carve-up per warp
    int off = kGridBytes;
    (void)stats_level;
    P.list_off = off;
    off += kMaxList * 4;
    P.bits_off = off;
    off += ((P.bits_words * 4 + 15) / 16) * 16 + 16;
    P.warp_smem_bytes = off;
    return CTF_OK;
}

extern "C" int ctf_create(const ctf_config_t* cfg, int64_t num_envs, int device, uint64_t seed, uint64_t env_id_base,
                          int stats_level, int obs_dtype, ctf_handle_t* out) {
    if (!cfg || !out) return fail(CTF_ERR_INVALID, "null argument");
    if (num_envs < 1) return fail(CTF_ERR_INVALID, "num_envs must be >= 1");
    if (stats_level < 0 || stats_level > 2) return fail(CTF_ERR_INVALID, "stats_level must be 0, 1 or 2");
    if (env_id_base + (uint64_t)num_envs > 0x100000000ull) return fail(CTF_ERR_INVALID, "global env ids must fit 32 bits");
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0)
        return fail(CTF_ERR_NO_DEVICE, "no CUDA device: the step path has no CPU fallback");
    if (device < 0 || device >= n_dev) return fail(CTF_ERR_INVALID, "device index out of range");
    ctf_env* h = new (std::nothrow) ctf_env();
    if (!h) return fail(CTF_ERR_INVALID, "out of host memory");
    int rc = build_plan(*cfg, stats_level, obs_dtype, h->plan);
    if (rc != CTF_OK) { delete h; return rc; }
    h->cfg = *cfg; h->B = num_envs; h->device = device; h->stats_level = stats_level; h->obs_dtype = obs_dtype;
    h->seed = seed; h->env_id_base = env_id_base;
    const size_t smem_unpadded = (obs_dtype == CTF_OBS_U8 ? kLutBytes<uint8_t> : 0) + (size_t)h->plan.warp_smem_bytes * kWarpsPerCta;
    h->smem_bytes = smem_unpadded;
    DeviceGuard guard(device);
    cudaError_t e = guard.err;
    if (e == cudaSuccess) e = cudaMalloc(&h->faults, sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMemset(h->faults, 0, sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMalloc(&h->actions_stage, (size_t)num_envs * cfg->n_agents);
    if (e == cudaSuccess) e = cudaMalloc(&h->rewards_stage, (size_t)num_envs * cfg->n_agents * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&h->dones_stage, (size_t)num_envs);
    int n_sm = 0;
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device);
    // Resident CTAs per SM of the warp-per-env kernels.  Registers allow 9 (36 warps); when the step is bound by the
    // observation stream, FEWER concurrent streams write faster (8_arena float32 B = 65536: 9 -> 1.001 ms, 7 -> 0.989,
    // 5 -> 0.980, 4 -> 0.982; 7_gridlocked 0.551 -> 0.536; bf16 0.526 -> 0.516), when it is bound by the env logic they
    // are slower (uint8 0.283 -> 0.347, 0_the_split 0.174 -> 0.229): profiles/r02_ab_residency*.log.  So blocks of
    // >= 6 KB per agent run with 5 CTAs per SM when there are many waves of them, and with the cap in 5..9 that fills
    // the last wave best when there are few (B = 16384: 7).  The cap is applied by padding dynamic shared memory.
    //
    // Into compressed memory (ctf_compressible_alloc, DESIGN §4) the mostly-zero stream moves far fewer DRAM bytes and
    // the env logic weighs more, so more resident CTAs win there (profiles/r05_residency_compressed.log, ms per step by
    // cap 5 / 7 / 9): 8_arena bf16 B = 65536 0.471 / 0.428 / 0.416, 7_gridlocked float32 0.507 / 0.492 / 0.484, at
    // B = 16384 bf16 0.135 / 0.123 / 0.119 and 7_gridlocked 0.151 / 0.136 / 0.132.  Only the 12.6 KB float32 blocks of
    // 8_arena stay write-bound enough to prefer 7 (0.832 / 0.822 / 0.831; B = 16384 0.242 / 0.226 / 0.230).  So on a
    // compressed buffer the cap is 7 for blocks of >= 12 KB per agent and 9 (what registers allow) below.  The launch picks the
    // padding from where outputs.obs lies (obs_in_compressed_memory).
    const size_t block_bytes = (size_t)h->plan.C * h->plan.GG * (obs_dtype == CTF_OBS_F32 ? 4 : (obs_dtype == CTF_OBS_U8 ? 1 : 2));
    h->smem_bytes_comp = h->smem_bytes;
    if (n_sm > 0 && block_bytes >= 6000) {
        const double ctas_per_sm_total = (double)((num_envs + kWarpsPerCta - 1) / kWarpsPerCta) / n_sm;
        int cap = 5;
        if (ctas_per_sm_total < 64.0) {
            double best = -1.0;
            for (int c = 5; c <= 9; ++c) {   // fill of the last wave; ties go to the smaller cap
                const double waves = ctas_per_sm_total / c, full = (double)(long long)(waves + 0.999999);
                const double fill = full > 0 ? waves / full : 0.0;
                if (fill > best + 1e-9) { best = fill; cap = c; }
            }
        }
        const size_t want = (size_t)(227 * 1024) / (size_t)cap - 1024;
        if (want > h->smem_bytes) h->smem_bytes = want;
        const size_t want_comp = (size_t)(227 * 1024) / (block_bytes >= 12 * 1024 ? 7 : 9) - 1024;
        if (want_comp > h->smem_bytes_comp) h->smem_bytes_comp = want_comp;
    }
    // Delta writes (ctf_bind_obs_record) store ~1.3 % of the sectors, so the step is bound by the env logic and the
    // record stream, not by the store stream: the cap is CTF_DELTA_CTAS_PER_SM on plain and compressed memory alike
    // (the sweep of tools/obs_delta_bench.py, profiles/r10_obs_delta.log).
    h->smem_bytes_delta = std::max(smem_unpadded, (size_t)(227 * 1024) / CTF_DELTA_CTAS_PER_SM - 1024);
    // The attribute is per kernel, not per handle: give every kernel a ceiling that covers any handle's launch (another
    // handle with a smaller footprint must not lower it under this one's), not this handle's own size.
    const int smem = h->smem_bytes > 100 * 1024 ? (int)h->smem_bytes : 100 * 1024;
#define CTF_SET_SMEM(K, BYTES) if (e == cudaSuccess) e = cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, BYTES)
#define CTF_SET_SMEM_T(T)                                                                                       \
    CTF_SET_SMEM((k_step<T, false, false, false>), smem); CTF_SET_SMEM((k_step<T, true, false, false>), smem); \
    CTF_SET_SMEM((k_step<T, false, true, false>), smem); CTF_SET_SMEM((k_step<T, true, true, false>), smem);   \
    CTF_SET_SMEM((k_step<T, false, false, true>), smem); CTF_SET_SMEM((k_step<T, true, false, true>), smem);   \
    CTF_SET_SMEM((k_step<T, false, true, true>), smem); CTF_SET_SMEM((k_step<T, true, true, true>), smem);     \
    CTF_SET_SMEM((k_reset<T, false>), smem); CTF_SET_SMEM((k_reset<T, true>), smem); CTF_SET_SMEM((k_observe<T>), smem); \
    CTF_SET_SMEM((k_unpack<T>), smem)
    CTF_SET_SMEM_T(float); CTF_SET_SMEM_T(uint8_t); CTF_SET_SMEM_T(__half); CTF_SET_SMEM_T(__nv_bfloat16);
    // A trunk kernel's dynamic shared memory ceiling (per kernel, so it covers every plan), then how many of its CTAs
    // this plan's launch fits on the device at once (at least one per SM; no query without a trunk, G < 5)
    auto trunk_ctas = [&](auto kernel, int threads, int ceiling, size_t smem_bytes) {
        CTF_SET_SMEM(kernel, ceiling);
        int per_sm = 0;
        if (e == cudaSuccess && h->plan.G >= 5)
            e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem_bytes);
        return (per_sm > 0 ? per_sm : 1) * (n_sm > 0 ? n_sm : 1);
    };
    TrunkGeometry tg;
    trunk_layout(h->plan, tg, h->trunk_smem_bytes);
    TrunkBwdArgs ba;
    trunk_bwd_layout(h->plan, ba, h->bwd_smem_bytes);
    // k_policy_trunk needs at most 94 KB (G = 16, C = 14)
    h->trunk_ctas = trunk_ctas(k_policy_trunk<1, 1>, kTrunkThreads, 100 * 1024, h->trunk_smem_bytes);
    h->grouped_ctas = trunk_ctas(k_policy_trunk<CTF_GROUPED_MAX_POLICIES, CTF_GROUPED_MAX_SEGMENTS>, kTrunkThreads,
                                 100 * 1024, h->trunk_smem_bytes);
    // k_policy_trunk_backward needs at most 46 KB (G = 16, C = 14)
    h->bwd_ctas = trunk_ctas(k_policy_trunk_backward, kBwdThreads, 64 * 1024, h->bwd_smem_bytes);
#undef CTF_SET_SMEM_T
#undef CTF_SET_SMEM
    if (e != cudaSuccess) {
        fail(CTF_ERR_CUDA, "ctf_create: %s", cudaGetErrorString(e));
        cudaFree(h->faults); cudaFree(h->actions_stage); cudaFree(h->rewards_stage); cudaFree(h->dones_stage);
        delete h;
        return CTF_ERR_CUDA;
    }
    *out = h;
    return CTF_OK;
}

extern "C" int ctf_destroy(ctf_handle_t h) {
    if (!h) return CTF_OK;
    DeviceGuard guard(h->device);
    cudaFree(h->faults); cudaFree(h->actions_stage); cudaFree(h->rewards_stage); cudaFree(h->dones_stage);
    delete h;
    return CTF_OK;
}

extern "C" int ctf_get_sizes(ctf_handle_t h, ctf_sizes_t* s) {
    if (!h || !s) return fail(CTF_ERR_INVALID, "null argument");
    const DevPlan& P = h->plan;
    const size_t B = (size_t)h->B, elem = h->obs_dtype == CTF_OBS_F32 ? 4 : (h->obs_dtype == CTF_OBS_U8 ? 1 : 2);
    s->grid_stride = kGridBytes;
    s->grid_bytes = B * kGridBytes;
    s->agents_bytes = B * P.N * 8;
    s->envs_bytes = B * 16;
    s->hp_bytes = h->plan.hp_float ? B * P.N * sizeof(double) : 0;
    s->stats_bytes = h->stats_level > 0 ? B * CTF_N_METRICS * P.N * 4 : 0;
    s->visits_bytes = h->stats_level > 1 ? B * P.N * P.GG : 0;
    s->obs_bytes = B * P.E * elem;
    s->obs_bits_bytes = B * P.N * P.wpa * 4;
    s->bits_words_per_agent = (size_t)P.wpa;
    s->meta_bytes = B * P.N * P.M * 4;
    s->rewards_bytes = B * P.N * 4;
    s->dones_bytes = B;
    s->obs_elems_per_env = (size_t)P.E;
    s->meta_elems_per_env = (size_t)P.N * P.M;
    return CTF_OK;
}

// [a, a + a_bytes) and [b, b + b_bytes) share a byte
static bool overlaps(const void* a, size_t a_bytes, const void* b, size_t b_bytes) {
    const uintptr_t x = reinterpret_cast<uintptr_t>(a), y = reinterpret_cast<uintptr_t>(b);
    return x < y + b_bytes && y < x + a_bytes;
}

extern "C" int ctf_obs_record_size(ctf_handle_t h, size_t* record_bytes) {
    if (!h || !record_bytes) return fail(CTF_ERR_INVALID, "null argument");
    *record_bytes = (size_t)h->B * h->plan.bits_words * sizeof(uint32_t);
    return CTF_OK;
}

extern "C" int ctf_bind_obs_record(ctf_handle_t h, const void* obs, uint32_t* record, uint32_t* record_epoch,
                                   const uint32_t* epoch) {
    if (!h) return fail(CTF_ERR_INVALID, "null handle");
    if (!obs) {
        h->rec_obs = nullptr; h->record = nullptr; h->record_epoch = nullptr; h->epoch = nullptr;
        return CTF_OK;
    }
    if (!record || !record_epoch || !epoch)
        return fail(CTF_ERR_INVALID, "ctf_bind_obs_record: record, record_epoch and epoch must not be null");
    if ((reinterpret_cast<uintptr_t>(record) & 15) || (reinterpret_cast<uintptr_t>(record_epoch) & 3) ||
        (reinterpret_cast<uintptr_t>(epoch) & 3))
        return fail(CTF_ERR_INVALID, "ctf_bind_obs_record: record must be 16-byte, record_epoch and epoch 4-byte aligned");
    const size_t elem = h->obs_dtype == CTF_OBS_F32 ? 4 : (h->obs_dtype == CTF_OBS_U8 ? 1 : 2);
    const size_t obs_bytes = (size_t)h->B * h->plan.E * elem, rec_bytes = (size_t)h->B * h->plan.bits_words * 4;
    const size_t ep_bytes = (size_t)h->B * 4;
    if (overlaps(obs, obs_bytes, record, rec_bytes) || overlaps(obs, obs_bytes, record_epoch, ep_bytes) ||
        overlaps(obs, obs_bytes, epoch, 4) || overlaps(record, rec_bytes, record_epoch, ep_bytes) ||
        overlaps(record, rec_bytes, epoch, 4) || overlaps(record_epoch, ep_bytes, epoch, 4))
        return fail(CTF_ERR_INVALID, "ctf_bind_obs_record: obs, record, record_epoch and epoch must not overlap");
    h->rec_obs = obs; h->record = record; h->record_epoch = record_epoch; h->epoch = epoch;
    return CTF_OK;
}

static int make_launch(ctf_handle_t h, const ctf_state_t& st, const ctf_outputs_t& out, Launch& L) {
    if (!st.grid || !st.agents || !st.envs) return fail(CTF_ERR_INVALID, "state.grid/agents/envs must not be null");
    if (h->stats_level > 0 && !st.stats) return fail(CTF_ERR_INVALID, "state.stats is null but the handle was created with stats");
    if (h->stats_level > 1 && !st.visits) return fail(CTF_ERR_INVALID, "state.visits is null but the handle was created with visitation maps");
    if ((reinterpret_cast<uintptr_t>(st.grid) & 15) || (reinterpret_cast<uintptr_t>(st.envs) & 15) ||
        (reinterpret_cast<uintptr_t>(st.agents) & 7))
        return fail(CTF_ERR_INVALID, "state buffers must be 16-byte aligned");
    if (reinterpret_cast<uintptr_t>(out.meta) & 15) return fail(CTF_ERR_INVALID, "outputs.meta must be 16-byte aligned");
    memset(&L, 0, sizeof(L));
    L.grid = st.grid; L.agents = reinterpret_cast<unsigned long long*>(st.agents); L.envs = reinterpret_cast<uint4*>(st.envs);
    if (h->plan.hp_float && (!st.hp || (reinterpret_cast<uintptr_t>(st.hp) & 7)))
        return fail(CTF_ERR_INVALID, "state.hp (8-byte aligned [B][N] doubles) is required when cfg.hp_float is set");
    L.hp = h->plan.hp_float ? st.hp : nullptr;
    L.stats = h->stats_level > 0 ? st.stats : nullptr;
    L.visits = h->stats_level > 1 ? st.visits : nullptr;
    L.obs = out.obs; L.obs_bits = out.obs_bits; L.meta = out.meta; L.rewards = out.rewards; L.dones = out.dones;
    L.faults = h->faults;
    if (out.obs && out.obs == h->rec_obs) {
        L.record = h->record; L.record_epoch = h->record_epoch; L.epoch = h->epoch;
    }
    L.B = h->B;
    L.seed_lo = (uint32_t)(h->seed & 0xFFFFFFFFu); L.seed_hi = (uint32_t)(h->seed >> 32);
    L.env_id_base = (uint32_t)h->env_id_base;
    return CTF_OK;
}

static unsigned grid_dim(long long B) { return (unsigned)((B + kWarpsPerCta - 1) / kWarpsPerCta); }

// Dynamic shared memory of a warp-per-env launch that writes `obs`: the residency cap depends on whether the buffer
// lies in compressed memory (ctf_create).  The answer is cached per pointer, so a step with the same buffer costs one
// comparison.
static size_t launch_smem(ctf_handle_t h, const void* obs) {
    if (!obs) return h->smem_bytes;
    if (obs != h->obs_seen) {
        int comp = 0;
        if (ctf_mem_is_compressed(obs, &comp) != CTF_OK) comp = 0;
        h->obs_seen = obs;
        h->obs_seen_comp = comp != 0;
    }
    return h->obs_seen_comp ? h->smem_bytes_comp : h->smem_bytes;
}

// calls f(T{}) with the observation element type of the handle
template <typename F>
static void with_obs_type(int obs_dtype, F&& f) {
    switch (obs_dtype) {
        case CTF_OBS_F32: f(float{}); break;
        case CTF_OBS_U8: f(uint8_t{}); break;
        case CTF_OBS_F16: f(__half{}); break;
        default: f(__nv_bfloat16{}); break;
    }
}

extern "C" int ctf_reset(ctf_handle_t h, ctf_state_t st, ctf_outputs_t out, int first, void* stream) {
    if (!h) return fail(CTF_ERR_INVALID, "null handle");
    Launch L;
    int rc = make_launch(h, st, out, L);
    if (rc != CTF_OK) return rc;
    L.first_reset = first ? 1 : 0;
    DeviceGuard guard(h->device);
    CTF_CUDA(guard.err);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const bool stats = h->stats_level > 0;
    const size_t smem = launch_smem(h, out.obs);
    with_obs_type(h->obs_dtype, [&](auto tag) {
        using T = decltype(tag);
        if (stats) k_reset<T, true><<<grid_dim(h->B), kThreads, smem, s>>>(h->plan, L);
        else k_reset<T, false><<<grid_dim(h->B), kThreads, smem, s>>>(h->plan, L);
    });
    CTF_CUDA(cudaGetLastError());
    return CTF_OK;
}

static int launch_step(ctf_handle_t h, const Launch& L, cudaStream_t s) {
    const bool stats = h->stats_level > 0;
    const bool hpf = h->plan.hp_float != 0;
    const size_t smem = L.record ? h->smem_bytes_delta : launch_smem(h, L.obs);
    with_obs_type(h->obs_dtype, [&](auto tag) {
        using T = decltype(tag);
        auto launch = [&](auto stats_c, auto hpf_c) {
            constexpr bool S = decltype(stats_c)::value, F = decltype(hpf_c)::value;
            if (L.record) k_step<T, S, F, true><<<grid_dim(h->B), kThreads, smem, s>>>(h->plan, L);
            else k_step<T, S, F, false><<<grid_dim(h->B), kThreads, smem, s>>>(h->plan, L);
        };
        if (stats) { if (hpf) launch(std::true_type{}, std::true_type{}); else launch(std::true_type{}, std::false_type{}); }
        else { if (hpf) launch(std::false_type{}, std::true_type{}); else launch(std::false_type{}, std::false_type{}); }
    });
    CTF_CUDA(cudaGetLastError());
    return CTF_OK;
}

extern "C" int ctf_step(ctf_handle_t h, ctf_state_t st, const uint8_t* actions, ctf_outputs_t out, void* stream) {
    if (!h) return fail(CTF_ERR_INVALID, "null handle");
    if (!actions) return fail(CTF_ERR_INVALID, "actions must not be null");
    Launch L;
    int rc = make_launch(h, st, out, L);
    if (rc != CTF_OK) return rc;
    L.actions = actions;
    DeviceGuard guard(h->device);
    CTF_CUDA(guard.err);
    return launch_step(h, L, static_cast<cudaStream_t>(stream));
}

extern "C" int ctf_observe(ctf_handle_t h, ctf_state_t st, const uint8_t* reverse_flags, ctf_outputs_t out, void* stream) {
    if (!h) return fail(CTF_ERR_INVALID, "null handle");
    Launch L;
    int rc = make_launch(h, st, out, L);
    if (rc != CTF_OK) return rc;
    if (reverse_flags) {
        uint32_t m = 0x100u;
        for (int i = 0; i < h->plan.N; ++i) m |= (reverse_flags[i] ? 1u : 0u) << i;
        L.rev_override = m;
    }
    DeviceGuard guard(h->device);
    CTF_CUDA(guard.err);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t smem = launch_smem(h, out.obs);
    with_obs_type(h->obs_dtype, [&](auto tag) {
        k_observe<decltype(tag)><<<grid_dim(h->B), kThreads, smem, s>>>(h->plan, L);
    });
    CTF_CUDA(cudaGetLastError());
    return CTF_OK;
}

extern "C" int ctf_unpack_obs(ctf_handle_t h, const uint32_t* packed, void* out, int out_dtype, int64_t n_agent_blocks,
                              void* stream) {
    if (!h || !packed || !out) return fail(CTF_ERR_INVALID, "null argument");
    if (out_dtype < CTF_OBS_F32 || out_dtype > CTF_OBS_BF16) return fail(CTF_ERR_INVALID, "unknown obs dtype");
    if (n_agent_blocks < 0) return fail(CTF_ERR_INVALID, "negative block count");
    if (n_agent_blocks == 0) return CTF_OK;
    DeviceGuard guard(h->device);
    CTF_CUDA(guard.err);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int nbits = h->plan.C * h->plan.GG, wpa = h->plan.wpa;
    const int elem = out_dtype == CTF_OBS_F32 ? 4 : (out_dtype == CTF_OBS_U8 ? 1 : 2);
    int chunk = (48 * 1024) / (nbits * elem);    // ~48 KB of output per CTA (12 .. 384 KB swept: profiles/r02_unpack_chunk_sweep.log)
    chunk = chunk < 1 ? 1 : (chunk > 64 ? 64 : chunk);
    while (chunk > 1 && ((size_t)(chunk * nbits) / 8 + (size_t)chunk * wpa * 4) > 40 * 1024) --chunk;   // static shared-memory budget
    const int bits_words = (((chunk * nbits + 128 + 31) / 32 + 1) + 15) / 16 * 16;
    const unsigned grid = (unsigned)((n_agent_blocks + chunk - 1) / chunk);
    size_t smem = ((size_t)bits_words + (size_t)chunk * wpa) * sizeof(uint32_t) + (out_dtype == CTF_OBS_U8 ? kLutBytes<uint8_t> : 0);
    // like k_step: fewer resident CTAs = fewer concurrent write streams (profiles/r02_unpack_residency.log)
    // float32 6 777 -> 6 838 GB/s and bf16 6 600 -> 6 703 at 5 CTAs per SM, uint8 (issue-bound) 6 365 -> 5 239: capped for >= 2-byte elements
    if (elem >= 2) {
        const size_t want = (size_t)(227 * 1024) / 5 - 1024;
        if (want > smem) smem = want;
    }
    with_obs_type(out_dtype, [&](auto tag) {
        using T = decltype(tag);
        k_unpack<T><<<grid, kUnpackThreads, smem, s>>>(packed, static_cast<T*>(out), n_agent_blocks, nbits, wpa, chunk, bits_words);
    });
    CTF_CUDA(cudaGetLastError());
    return CTF_OK;
}

// The checks the three trunk entry points share.  `fn` names the entry point in the error messages.
//
// The plan has a trunk (G >= 5), the packed blocks are addressed with agents_per_env >= 1 and n_envs >= 0, and a
// feature row holds 32*(G-4)^2 + M values with a stride that keeps its 16-byte stores aligned.
static int check_trunk_geometry(const char* fn, const DevPlan& P, int64_t n_envs, int agents_per_env,
                                int64_t feature_stride) {
    if (P.G < 5) return fail(CTF_ERR_INVALID, "%s: the policy needs grid_size >= 5 (two valid 3x3 convolutions)", fn);
    if (agents_per_env < 1) return fail(CTF_ERR_INVALID, "%s: agents_per_env must be >= 1", fn);
    if (n_envs < 0) return fail(CTF_ERR_INVALID, "%s: negative n_envs", fn);
    const long long k1 = 32LL * (P.G - 4) * (P.G - 4) + P.M;
    if (feature_stride < k1 || (feature_stride & 7))
        return fail(CTF_ERR_INVALID, "%s: feature_stride must be a multiple of 8 and >= 32*(G-4)^2 + M", fn);
    return CTF_OK;
}

// 1..8 agent ids, each < agents_per_env; `k_name` is how the entry point calls k
static int check_agent_ids(const char* fn, const char* k_name, const uint8_t* agent_ids, int k, int agents_per_env) {
    if (k < 1 || k > CTF_MAX_AGENTS) return fail(CTF_ERR_INVALID, "%s: %s must be in 1..8", fn, k_name);
    for (int j = 0; j < k; ++j)
        if (agent_ids[j] >= agents_per_env) return fail(CTF_ERR_INVALID, "%s: an agent id is >= agents_per_env", fn);
    return CTF_OK;
}

// No weight pointer is null, and the ones the kernel reads are aligned for its loads: conv1_w 16 bytes, the fp32
// biases 4.  The forward kernels read conv2_w (8 bytes) and conv2_b; the backward reads conv1 only from `w` (its conv2
// comes transposed, in a buffer of its own).
static int check_trunk_weights(const char* fn, const ctf_policy_weights_t& w, bool reads_conv2) {
    if (!w.conv1_w || !w.conv1_b || !w.conv2_w || !w.conv2_b) return fail(CTF_ERR_INVALID, "%s: null weight pointer", fn);
    if ((reinterpret_cast<uintptr_t>(w.conv1_w) & 15) || (reinterpret_cast<uintptr_t>(w.conv1_b) & 3) ||
        (reads_conv2 && ((reinterpret_cast<uintptr_t>(w.conv2_w) & 7) || (reinterpret_cast<uintptr_t>(w.conv2_b) & 3))))
        return fail(CTF_ERR_INVALID, "%s: misaligned weights", fn);
    return CTF_OK;
}

// Fills the argument block of one trunk launch from checked arguments with at least one sample and launches
// k_policy_trunk with that block's table sizes on at most `ctas` CTAs.
template <int kMaxPolicies, int kMaxSegments>
static void launch_trunk_table(TrunkLaunch<kMaxPolicies, kMaxSegments>& A, const TrunkGeometry& geo,
                               const ctf_policy_weights_t* weights, int n_policies, const ctf_policy_segment_t* segments,
                               int n_segments, int agents_per_env, int ctas, size_t smem, cudaStream_t stream) {
    memset(&A, 0, sizeof(A));
    A.geo = geo;
    for (int p = 0; p < n_policies; ++p) {
        const ctf_policy_weights_t& w = weights[p];
        A.w[p].conv1_w = w.conv1_w; A.w[p].conv1_b = w.conv1_b;
        A.w[p].conv2_w = static_cast<const uint2*>(w.conv2_w); A.w[p].conv2_b = w.conv2_b;
    }
    long long tiles = 0;
    for (int i = 0; i < n_segments; ++i) {
        const ctf_policy_segment_t& g = segments[i];
        TrunkSegment& T = A.seg[i];
        T.blk_begin = g.env_begin * agents_per_env;
        T.row_begin = g.out_row;
        T.n_samples = g.n_envs * g.k;
        T.tile_begin = tiles;
        T.policy = g.policy;
        T.k = g.k;
        for (int j = 0; j < g.k; ++j) T.ids[j] = g.agent_ids[j];
        tiles += (T.n_samples + kTrunkWarps - 1) / kTrunkWarps;
    }
    A.n_tiles = tiles;
    A.n_segments = n_segments;
    const unsigned grid = (unsigned)(tiles < ctas ? tiles : ctas);
    k_policy_trunk<kMaxPolicies, kMaxSegments><<<grid, kTrunkThreads, smem, stream>>>(A);
}

// The forward trunk of both entry points: checks every argument, then launches k_policy_trunk<1, 1> for one policy and
// one segment, the grouped instantiation otherwise.  Errors name the entry point `fn` and call a segment's k `k_name`.
static int launch_trunk(const char* fn, const char* k_name, ctf_handle_t h, const ctf_policy_weights_t* weights,
                        int n_policies, const ctf_policy_segment_t* segments, int n_segments, const uint32_t* packed,
                        const float* meta, int64_t n_envs, int agents_per_env, void* features, int64_t feature_stride,
                        int64_t n_rows, void* stream) {
    const DevPlan& P = h->plan;
    int rc = check_trunk_geometry(fn, P, n_envs, agents_per_env, feature_stride);
    if (rc != CTF_OK) return rc;
    if (n_policies < 1 || n_policies > CTF_GROUPED_MAX_POLICIES)
        return fail(CTF_ERR_INVALID, "%s: n_policies must be in 1..CTF_GROUPED_MAX_POLICIES (64)", fn);
    if (n_segments < 1 || n_segments > CTF_GROUPED_MAX_SEGMENTS)
        return fail(CTF_ERR_INVALID, "%s: n_segments must be in 1..CTF_GROUPED_MAX_SEGMENTS (512)", fn);
    if (n_rows < 0) return fail(CTF_ERR_INVALID, "%s: negative n_rows", fn);
    if (reinterpret_cast<uintptr_t>(features) & 15) return fail(CTF_ERR_INVALID, "%s: features must be 16-byte aligned", fn);
    if ((reinterpret_cast<uintptr_t>(packed) & 3) || (reinterpret_cast<uintptr_t>(meta) & 3))
        return fail(CTF_ERR_INVALID, "%s: misaligned inputs", fn);
    for (int p = 0; p < n_policies; ++p)
        if ((rc = check_trunk_weights(fn, weights[p], true)) != CTF_OK) return rc;
    int order[CTF_GROUPED_MAX_SEGMENTS];
    int n_busy = 0;
    for (int i = 0; i < n_segments; ++i) {
        const ctf_policy_segment_t& g = segments[i];
        if (g.policy < 0 || g.policy >= n_policies)
            return fail(CTF_ERR_INVALID, "%s: a segment's policy index is out of range", fn);
        if ((rc = check_agent_ids(fn, k_name, g.agent_ids, g.k, agents_per_env)) != CTF_OK) return rc;
        if (g.env_begin < 0 || g.n_envs < 0 || g.env_begin > n_envs || g.n_envs > n_envs - g.env_begin)
            return fail(CTF_ERR_INVALID, "%s: a segment's env range is outside [0, n_envs)", fn);
        const long long ns = g.n_envs * g.k;
        if (g.out_row < 0 || g.out_row > n_rows || ns > n_rows - g.out_row)
            return fail(CTF_ERR_INVALID, "%s: a segment's output rows are outside [0, n_rows)", fn);
        if (ns > 0) order[n_busy++] = i;
    }
    // no two segments may write the same row (the result would depend on the schedule)
    std::sort(order, order + n_busy, [&](int a, int b) { return segments[a].out_row < segments[b].out_row; });
    for (int i = 1; i < n_busy; ++i) {
        const ctf_policy_segment_t& prev = segments[order[i - 1]];
        if (prev.out_row + prev.n_envs * prev.k > segments[order[i]].out_row)
            return fail(CTF_ERR_INVALID, "%s: the output rows of two segments overlap", fn);
    }
    if (n_busy == 0) return CTF_OK;
    TrunkGeometry geo;
    size_t smem = 0;
    trunk_layout(P, geo, smem);
    geo.packed = packed; geo.meta = meta; geo.features = static_cast<__nv_bfloat16*>(features);
    geo.stride = feature_stride; geo.ape = agents_per_env;
    DeviceGuard guard(h->device);
    CTF_CUDA(guard.err);
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (n_policies == 1 && n_segments == 1) {
        TrunkLaunchOne A;
        launch_trunk_table(A, geo, weights, n_policies, segments, n_segments, agents_per_env, h->trunk_ctas, smem, s);
    } else {
        // the grouped argument block is large (about 26 KB): keep it off the caller's stack
        static thread_local TrunkLaunchGrouped A;
        launch_trunk_table(A, geo, weights, n_policies, segments, n_segments, agents_per_env, h->grouped_ctas, smem, s);
    }
    CTF_CUDA(cudaGetLastError());
    return CTF_OK;
}

extern "C" int ctf_policy_features(ctf_handle_t h, const ctf_policy_weights_t* w, const uint32_t* packed, const float* meta,
                                   int64_t n_envs, int agents_per_env, const uint8_t* agent_ids, int k, void* features,
                                   int64_t feature_stride, void* stream) {
    const char* fn = "ctf_policy_features";
    if (!h || !w || !packed || !meta || !agent_ids || !features) return fail(CTF_ERR_INVALID, "%s: null argument", fn);
    // one segment over every env whose sample s is feature row s; launch_trunk rejects a k outside 1..8 (the ids are
    // copied only for a k in range, and n_rows stays >= 0 so that it is k that the error names)
    ctf_policy_segment_t seg = {0, n_envs, 0, 0, k, {}};
    if (k >= 1 && k <= CTF_MAX_AGENTS) memcpy(seg.agent_ids, agent_ids, k);
    const int64_t n_rows = k > 0 ? n_envs * k : 0;
    return launch_trunk(fn, "k", h, w, 1, &seg, 1, packed, meta, n_envs, agents_per_env, features, feature_stride, n_rows,
                        stream);
}

extern "C" int ctf_policy_features_grouped(ctf_handle_t h, const ctf_policy_weights_t* weights, int n_policies,
                                           const ctf_policy_segment_t* segments, int n_segments, const uint32_t* packed,
                                           const float* meta, int64_t n_envs, int agents_per_env, void* features,
                                           int64_t feature_stride, int64_t n_rows, void* stream) {
    const char* fn = "ctf_policy_features_grouped";
    if (!h || !weights || !segments || !packed || !meta || !features) return fail(CTF_ERR_INVALID, "%s: null argument", fn);
    return launch_trunk(fn, "a segment's k", h, weights, n_policies, segments, n_segments, packed, meta, n_envs,
                        agents_per_env, features, feature_stride, n_rows, stream);
}

extern "C" int ctf_policy_trunk_ctas(ctf_handle_t h, int* trunk_ctas, int* grouped_ctas) {
    if (!h || !trunk_ctas || !grouped_ctas) return fail(CTF_ERR_INVALID, "ctf_policy_trunk_ctas: null argument");
    *trunk_ctas = h->trunk_ctas;
    *grouped_ctas = h->grouped_ctas;
    return CTF_OK;
}

extern "C" int ctf_policy_grad_workspace_size(ctf_handle_t h, size_t* bytes) {
    if (!h || !bytes) return fail(CTF_ERR_INVALID, "ctf_policy_grad_workspace_size: null argument");
    if (h->plan.G < 5)
        return fail(CTF_ERR_INVALID, "ctf_policy_grad_workspace_size: the policy needs grid_size >= 5 (two valid 3x3 convolutions)");
    *bytes = (size_t)h->bwd_ctas * grad_count(h->plan.C) * sizeof(float);
    return CTF_OK;
}

extern "C" int ctf_policy_features_backward(ctf_handle_t h, const ctf_policy_weights_t* w, const void* conv2_w_t,
                                            const uint32_t* packed, int64_t n_envs, int agents_per_env,
                                            const uint8_t* agent_ids, int k, const void* features,
                                            const void* grad_features, int64_t feature_stride, void* workspace,
                                            size_t workspace_bytes, const ctf_policy_grads_t* grads, void* stream) {
    const char* fn = "ctf_policy_features_backward";
    if (!h || !w || !conv2_w_t || !packed || !agent_ids || !features || !grad_features || !workspace || !grads)
        return fail(CTF_ERR_INVALID, "%s: null argument", fn);
    if (!grads->conv1_w || !grads->conv1_b || !grads->conv2_w || !grads->conv2_b)
        return fail(CTF_ERR_INVALID, "%s: null gradient pointer", fn);
    const DevPlan& P = h->plan;
    int rc = check_trunk_geometry(fn, P, n_envs, agents_per_env, feature_stride);
    if (rc == CTF_OK) rc = check_agent_ids(fn, "k", agent_ids, k, agents_per_env);
    if (rc == CTF_OK) rc = check_trunk_weights(fn, *w, false);
    if (rc != CTF_OK) return rc;
    if ((reinterpret_cast<uintptr_t>(features) & 15) || (reinterpret_cast<uintptr_t>(grad_features) & 15))
        return fail(CTF_ERR_INVALID, "%s: features and grad_features must be 16-byte aligned", fn);
    if ((reinterpret_cast<uintptr_t>(conv2_w_t) & 7) || (reinterpret_cast<uintptr_t>(packed) & 3) ||
        (reinterpret_cast<uintptr_t>(workspace) & 15) || (reinterpret_cast<uintptr_t>(grads->conv1_w) & 3) ||
        (reinterpret_cast<uintptr_t>(grads->conv1_b) & 3) || (reinterpret_cast<uintptr_t>(grads->conv2_w) & 3) ||
        (reinterpret_cast<uintptr_t>(grads->conv2_b) & 3))
        return fail(CTF_ERR_INVALID, "%s: misaligned conv2_w_t, inputs, workspace or gradients", fn);
    const int n_grad = grad_count(P.C);
    if (workspace_bytes < (size_t)h->bwd_ctas * n_grad * sizeof(float))
        return fail(CTF_ERR_INVALID, "%s: workspace smaller than ctf_policy_grad_workspace_size", fn);
    const long long n = (long long)n_envs * k;
    TrunkBwdArgs A;
    memset(&A, 0, sizeof(A));
    size_t smem = 0;
    trunk_bwd_layout(P, A, smem);
    A.conv1_w = w->conv1_w; A.conv1_b = w->conv1_b; A.conv2_wt = static_cast<const uint2*>(conv2_w_t);
    A.packed = packed;
    A.features = static_cast<const __nv_bfloat16*>(features);
    A.grad_features = static_cast<const __nv_bfloat16*>(grad_features);
    A.partial = static_cast<float*>(workspace);
    A.n_samples = n; A.stride = feature_stride; A.ape = agents_per_env; A.k = k;
    for (int j = 0; j < k; ++j) A.ids[j] = agent_ids[j];
    DeviceGuard guard(h->device);
    CTF_CUDA(guard.err);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    // one CTA per sample up to bwd_ctas: the partition of samples into rows, and so every sum, depends on n alone
    const int parts = (int)(n < h->bwd_ctas ? n : h->bwd_ctas);
    if (parts > 0) k_policy_trunk_backward<<<parts, kBwdThreads, smem, s>>>(A);
    const int total = 16 * P.C * 9 + 16 + 32 * 144 + 32;
    k_policy_grad_reduce<<<(total + 255) / 256, 256, 0, s>>>(A.partial, parts, P.C, grads->conv1_w, grads->conv1_b,
                                                             grads->conv2_w, grads->conv2_b);
    CTF_CUDA(cudaGetLastError());
    return CTF_OK;
}

extern "C" int ctf_stats_sum(ctf_handle_t h, ctf_state_t st, int64_t* stats_sum, void* stream) {
    if (!h || !stats_sum) return fail(CTF_ERR_INVALID, "null argument");
    if (h->stats_level == 0 || !st.stats) return fail(CTF_ERR_INVALID, "handle was created without statistics");
    DeviceGuard guard(h->device);
    CTF_CUDA(guard.err);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int ns = CTF_N_METRICS * h->plan.N;
    CTF_CUDA(cudaMemsetAsync(stats_sum, 0, sizeof(int64_t) * ns, s));
    const int threads = 832;  // 8 * 104: a multiple of ns for N = 8 (and >= ns for every N)
    const unsigned blocks = (unsigned)((h->B + 255) / 256 < 592 ? (h->B + 255) / 256 : 592);
    k_stats_sum<<<blocks ? blocks : 1, threads, 0, s>>>(st.stats, h->B, ns, reinterpret_cast<unsigned long long*>(stats_sum));
    CTF_CUDA(cudaGetLastError());
    return CTF_OK;
}

extern "C" int ctf_take_faults(ctf_handle_t h, void* stream, uint32_t* faults) {
    if (!h || !faults) return fail(CTF_ERR_INVALID, "null argument");
    DeviceGuard guard(h->device);
    CTF_CUDA(guard.err);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CTF_CUDA(cudaMemcpyAsync(faults, h->faults, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    CTF_CUDA(cudaMemsetAsync(h->faults, 0, sizeof(uint32_t), s));
    CTF_CUDA(cudaStreamSynchronize(s));
    return CTF_OK;
}

// device-visible alias of a pinned (page-locked, UVA-mapped) host buffer, or nullptr for pageable memory
static void* mapped_alias(const void* host_ptr) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, host_ptr) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    if (attr.type == cudaMemoryTypeHost && attr.devicePointer) return attr.devicePointer;
    return nullptr;
}

extern "C" int ctf_step_host(ctf_handle_t h, ctf_state_t st, const uint8_t* actions_host, ctf_outputs_t out,
                             float* rewards_host, uint8_t* dones_host, void* stream) {
    if (!h) return fail(CTF_ERR_INVALID, "null handle");
    if (!actions_host) return fail(CTF_ERR_INVALID, "actions_host must not be null");
    DeviceGuard guard(h->device);
    CTF_CUDA(guard.err);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t n = (size_t)h->B * h->plan.N;
    // Pinned host buffers are read / written by the kernel itself over PCIe (zero-copy): 8 B of actions in and
    // 33 B of rewards + done out per env ride along with the step instead of three serialized copies.
    // Pageable buffers go through the handle's staging buffers.
    uint8_t* a_dev = static_cast<uint8_t*>(mapped_alias(actions_host));
    float* r_dev = rewards_host ? static_cast<float*>(mapped_alias(rewards_host)) : nullptr;
    uint8_t* d_dev = dones_host ? static_cast<uint8_t*>(mapped_alias(dones_host)) : nullptr;
    const bool r_copy = rewards_host && !r_dev, d_copy = dones_host && !d_dev;
    if (r_dev) out.rewards = r_dev;
    else if (!out.rewards) out.rewards = h->rewards_stage;
    if (d_dev) out.dones = d_dev;
    else if (!out.dones) out.dones = h->dones_stage;
    Launch L;
    int rc = make_launch(h, st, out, L);
    if (rc != CTF_OK) return rc;
    if (a_dev) {
        L.actions = a_dev;
    } else {
        CTF_CUDA(cudaMemcpyAsync(h->actions_stage, actions_host, n, cudaMemcpyHostToDevice, s));
        L.actions = h->actions_stage;
    }
    rc = launch_step(h, L, s);
    if (rc != CTF_OK) return rc;
    if (r_copy) CTF_CUDA(cudaMemcpyAsync(rewards_host, out.rewards, n * sizeof(float), cudaMemcpyDeviceToHost, s));
    if (d_copy) CTF_CUDA(cudaMemcpyAsync(dones_host, out.dones, (size_t)h->B, cudaMemcpyDeviceToHost, s));
    CTF_CUDA(cudaStreamSynchronize(s));
    return CTF_OK;
}

// ctf_gae and ctf_gae_dones: checks every argument, then launches k_gae<dones != nullptr>.  `fn` names the entry point
// in the error messages.
static int launch_gae(const char* fn, ctf_handle_t h, const float* rewards, const float* values, const float* dones,
                      const float* next_value, float* advantages, float* returns, int64_t n_steps,
                      int64_t agents_per_step, int64_t n_envs, float gamma, float gamma_lambda, void* stream) {
    if (!h || !rewards || !values || !next_value || !advantages || !returns)
        return fail(CTF_ERR_INVALID, "%s: null argument", fn);
    if (n_steps < 1) return fail(CTF_ERR_INVALID, "%s: n_steps must be >= 1", fn);
    if (agents_per_step < 1 || agents_per_step > CTF_MAX_AGENTS)
        return fail(CTF_ERR_INVALID, "%s: agents_per_step must be in 1..CTF_MAX_AGENTS (8)", fn);
    if (n_envs < 1) return fail(CTF_ERR_INVALID, "%s: n_envs must be >= 1", fn);
    // the comparisons are false for NaN, so a NaN is rejected too
    if (!(gamma >= 0.f && gamma <= 1.f)) return fail(CTF_ERR_INVALID, "%s: gamma must be finite and in [0, 1]", fn);
    if (!(gamma_lambda >= 0.f && gamma_lambda <= 1.f))
        return fail(CTF_ERR_INVALID, "%s: gamma_lambda must be finite and in [0, 1]", fn);
    const long long cols = (long long)agents_per_step * n_envs;
    // one thread per column: the grid must stay below 2^31 CTAs, and the byte sizes must fit 64 bits
    if (n_envs > (1LL << 35) || n_steps > (1LL << 60) / cols)
        return fail(CTF_ERR_INVALID, "%s: n_steps * agents_per_step * n_envs is too large", fn);
    if ((reinterpret_cast<uintptr_t>(rewards) | reinterpret_cast<uintptr_t>(values) |
         reinterpret_cast<uintptr_t>(dones) | reinterpret_cast<uintptr_t>(next_value) |
         reinterpret_cast<uintptr_t>(advantages) | reinterpret_cast<uintptr_t>(returns)) & 3)
        return fail(CTF_ERR_INVALID, "%s: every buffer must be 4-byte aligned", fn);
    const size_t bytes = (size_t)(n_steps * cols) * sizeof(float), nv_bytes = (size_t)cols * sizeof(float);
    for (const float* out : {advantages, returns})
        if (overlaps(out, bytes, rewards, bytes) || overlaps(out, bytes, values, bytes) ||
            overlaps(out, bytes, next_value, nv_bytes) || (dones && overlaps(out, bytes, dones, bytes)))
            return fail(CTF_ERR_INVALID, "%s: an output overlaps an input", fn);
    if (overlaps(advantages, bytes, returns, bytes)) return fail(CTF_ERR_INVALID, "%s: advantages overlaps returns", fn);
    DeviceGuard guard(h->device);
    CTF_CUDA(guard.err);
    const unsigned grid = (unsigned)((cols + kGaeThreads - 1) / kGaeThreads);
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (dones)
        k_gae<true><<<grid, kGaeThreads, 0, s>>>(rewards, values, next_value, advantages, returns, n_steps, cols, gamma,
                                                 gamma_lambda, dones);
    else
        k_gae<false><<<grid, kGaeThreads, 0, s>>>(rewards, values, next_value, advantages, returns, n_steps, cols, gamma,
                                                  gamma_lambda, nullptr);
    CTF_CUDA(cudaGetLastError());
    return CTF_OK;
}

extern "C" int ctf_gae(ctf_handle_t h, const float* rewards, const float* values, const float* next_value,
                       float* advantages, float* returns, int64_t n_steps, int64_t agents_per_step, int64_t n_envs,
                       float gamma, float gamma_lambda, void* stream) {
    return launch_gae("ctf_gae", h, rewards, values, nullptr, next_value, advantages, returns, n_steps, agents_per_step,
                      n_envs, gamma, gamma_lambda, stream);
}

extern "C" int ctf_gae_dones(ctf_handle_t h, const float* rewards, const float* values, const float* dones,
                             const float* next_value, float* advantages, float* returns, int64_t n_steps,
                             int64_t agents_per_step, int64_t n_envs, float gamma, float gamma_lambda, void* stream) {
    if (!dones) return fail(CTF_ERR_INVALID, "ctf_gae_dones: null argument");
    return launch_gae("ctf_gae_dones", h, rewards, values, dones, next_value, advantages, returns, n_steps,
                      agents_per_step, n_envs, gamma, gamma_lambda, stream);
}

extern "C" int ctf_sample_actions(ctf_handle_t h, ctf_state_t state, const float* head, int64_t head_stride,
                                  const uint8_t* masked, const int64_t* flat_index, int64_t n_rows, uint64_t seed,
                                  uint8_t* actions, int64_t* action_out, float* logprob, float* entropy,
                                  void* stream) {
    if (!h || !state.envs || !head || !flat_index) return fail(CTF_ERR_INVALID, "ctf_sample_actions: null argument");
    if (n_rows < 0) return fail(CTF_ERR_INVALID, "ctf_sample_actions: n_rows must be >= 0");
    if (head_stride < 1 + CTF_N_ACTIONS)
        return fail(CTF_ERR_INVALID, "ctf_sample_actions: head_stride must be >= 10 (value, then 9 logits)");
    // one thread per row: the grid must stay below 2^31 CTAs, and the head's byte size must fit 64 bits
    if (n_rows > (1LL << 38) || (n_rows > 0 && head_stride > (1LL << 58) / n_rows))
        return fail(CTF_ERR_INVALID, "ctf_sample_actions: n_rows * head_stride is too large");
    if ((reinterpret_cast<uintptr_t>(state.envs) & 15) || (reinterpret_cast<uintptr_t>(head) & 3) ||
        (reinterpret_cast<uintptr_t>(flat_index) & 7) || (reinterpret_cast<uintptr_t>(action_out) & 7) ||
        (reinterpret_cast<uintptr_t>(logprob) & 3) || (reinterpret_cast<uintptr_t>(entropy) & 3))
        return fail(CTF_ERR_INVALID, "ctf_sample_actions: misaligned buffer (state.envs 16-byte, flat_index and "
                                     "action_out 8-byte, head, logprob and entropy 4-byte)");
    const size_t n = (size_t)n_rows, n_flat = (size_t)h->B * h->plan.N;
    // [pointer, bytes]: the inputs, then the outputs (absent ones have no bytes)
    const void* ptr[7] = {head, masked, flat_index, actions, action_out, logprob, entropy};
    const size_t bytes[7] = {n ? ((n - 1) * (size_t)head_stride + 1 + CTF_N_ACTIONS) * sizeof(float) : 0,
                             masked ? n : 0, n * sizeof(int64_t), actions ? n_flat : 0,
                             action_out ? n * sizeof(int64_t) : 0, logprob ? n * sizeof(float) : 0,
                             entropy ? n * sizeof(float) : 0};
    for (int o = 3; o < 7; ++o)
        for (int i = 0; i < o; ++i)
            if (bytes[o] && bytes[i] && overlaps(ptr[o], bytes[o], ptr[i], bytes[i]))
                return fail(CTF_ERR_INVALID, i < 3 ? "ctf_sample_actions: an output overlaps an input"
                                                   : "ctf_sample_actions: two outputs overlap");
    if (n_rows == 0) return CTF_OK;
    DeviceGuard guard(h->device);
    CTF_CUDA(guard.err);
    const unsigned grid = (unsigned)((n_rows + kSampleThreads - 1) / kSampleThreads);
    k_sample_actions<<<grid, kSampleThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        head, head_stride, masked, reinterpret_cast<const long long*>(flat_index), n_rows,
        reinterpret_cast<const uint4*>(state.envs), (long long)n_flat, h->plan.N, (uint32_t)h->env_id_base,
        (uint32_t)(seed & 0xFFFFFFFFu), (uint32_t)(seed >> 32), actions, reinterpret_cast<long long*>(action_out),
        logprob, entropy, h->faults);
    CTF_CUDA(cudaGetLastError());
    return CTF_OK;
}
