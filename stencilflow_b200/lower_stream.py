"""Streamed (temporally blocked) lowering: several chained operators in one pass over HBM.

What the reference builds out of FPGA shift registers and FIFOs -- every operator a processing
element holding a sliding window of its inputs (``stencilflow/stencil/intel_fpga.py:58-69,367-461``),
connected by delay buffers sized by ``compute_delay_buffer`` (``stencilflow/kernel_chain_graph.py:476-559``)
so that only program inputs and outputs touch off-chip memory (``generate_sdfg``,
``stencilflow/sdfg_generator.py:219-577``) -- becomes one CUDA kernel per fusion group:

* the group streams along the outermost dimension (i for 3-D programs, j for 2-D ones); a CTA owns a
  tile of the remaining dimension(s) including the halo the fused operators consume;
* planes of the group's input fields are staged into a shared-memory ring by TMA
  (``cp.async.bulk.tensor`` + mbarrier), ``PREFETCH`` steps ahead of their use;
* every field (group input or operator result) lives in a *register sliding window* over the streamed
  dimension: thread (warp, lane) owns R rows x V consecutive cells and keeps its own values of the
  last W planes, so taps at (dj, dk) = (0, 0) cost nothing;
* in-plane neighbours along the innermost dimension come from warp shuffles, neighbours along the
  row dimension from the adjacent warps through small shared-memory exchange rings (only the edge
  rows of each warp are published);
* operator A runs ``lag(A)`` planes behind the input stream -- the plane lags are the restriction of
  the reference's path-length recurrence to the streamed dimension with unit latency -- and one
  ``__syncthreads`` per streamed plane separates producers from consumers;
* boundary conditions are applied where a field is *produced*: cells outside the domain are set to
  the constant (or to -100000 for ``shrink``) the consumers would read, which is exactly what
  ``ExpandStencilCPU`` selects per tap (``stencilflow/stencil/cpu.py:73-102``).
"""

import collections
import hashlib
import math
import os
from typing import Dict, List, Optional, Tuple

from . import dtypes
from . import expr as ex
from .lower_cuda import (KernelSpec, LaunchSpec, LoweredProgram, _MATH_F32, _MATH_F64, ctype_of, value_literal,
                         literal)
from .stencil_op import JUNK_VAL, StencilOp, StencilProgram

SMEM_LIMIT = 227 * 1024
DEFAULT_SYNC = "cta"        # "pair": neighbour-only named barriers + per-warp TMA staging (see Geometry)
REG_SLACK = int(os.environ.get("SFB200_REG_SLACK", "0"))   # the estimate may exceed the per-thread limit by this much

STREAM_PRELUDE = r"""
// ---- streamed-kernel support (TMA + mbarrier, sm_100a) ----
struct __align__(64) CUtensorMap_st { unsigned long long opaque[16]; };
typedef CUtensorMap_st CUtensorMap;

__device__ __forceinline__ u32 sf_smem_addr(const void* p) {
    return (u32)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void sf_mbar_init(void* bar, u32 count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(sf_smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void sf_fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void sf_fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void sf_mbar_expect_tx(void* bar, u32 bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sf_smem_addr(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void sf_mbar_arrive(void* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(sf_smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void sf_mbar_wait(void* bar, u32 parity) {
    u32 addr = sf_smem_addr(bar);
    u32 done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
    }
}
__device__ __forceinline__ bool sf_elect_one() {
    u32 pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
// L2 eviction priorities (the encodings CUTLASS passes as TMA cache hints): SF_LOAD_HINT / SF_STORE_HINT are
// defined by the generator when a plan asks for them (input planes are re-read by the neighbouring tiles:
// keep them; results are written once: let them go first)
#define SF_L2_EVICT_FIRST 0x12F0000000000000ull
#define SF_L2_EVICT_LAST 0x14F0000000000000ull
__device__ __forceinline__ void sf_tma_load_3d(void* dst, const CUtensorMap* map, void* bar, int c0, int c1, int c2) {
#ifdef SF_LOAD_HINT
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;"
        ::"r"(sf_smem_addr(dst)), "l"(map), "r"(sf_smem_addr(bar)), "r"(c0), "r"(c1), "r"(c2), "l"(SF_LOAD_HINT)
        : "memory");
#else
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(sf_smem_addr(dst)), "l"(map), "r"(sf_smem_addr(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
#endif
}
__device__ __forceinline__ void sf_tma_load_2d(void* dst, const CUtensorMap* map, void* bar, int c0, int c1) {
#ifdef SF_LOAD_HINT
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(sf_smem_addr(dst)), "l"(map), "r"(sf_smem_addr(bar)), "r"(c0), "r"(c1), "l"(SF_LOAD_HINT)
        : "memory");
#else
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(sf_smem_addr(dst)), "l"(map), "r"(sf_smem_addr(bar)), "r"(c0), "r"(c1)
        : "memory");
#endif
}
#ifdef SF_STORE_HINT
#define SF_STG_V4F32 "st.global.L2::cache_hint.v4.f32 [%1], {%2, %3, %4, %5}, %6;"
#define SF_STG_V2F64 "st.global.L2::cache_hint.v2.f64 [%1], {%2, %3}, %4;"
#define SF_STG_V2F32 "st.global.L2::cache_hint.v2.f32 [%1], {%2, %3}, %4;"
#define SF_STG_HINT_ARG , "l"(SF_STORE_HINT)
#define SF_STG_HINT_ARG2 , "l"(SF_STORE_HINT)
#else
#define SF_STG_V2F32 "st.global.v2.f32 [%1], {%2, %3};"
#define SF_STG_HINT_ARG2
#define SF_STG_V4F32 "st.global.v4.f32 [%1], {%2, %3, %4, %5};"
#define SF_STG_V2F64 "st.global.v2.f64 [%1], {%2, %3};"
#define SF_STG_HINT_ARG
#endif
// ---- slab mode: edge planes of a result go to the neighbouring GPU's halo planes (peer stores over NVLink) ----
// Run by all threads of a CTA after it has streamed a segment: planes [p0, p1), rows [j0, j1), columns
// [k0, k1) of its own result -- just written, L2-resident -- are copied to the same cells of the
// neighbour's buffer, `delta` bytes away in the unified address space.  Doing this once per segment
// instead of next to the result stores keeps the streamed loop free of extra live registers.
__device__ __forceinline__ float4 sf_ldcg16(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ double2 sf_ldcg16(const double* p) { return __ldcg(reinterpret_cast<const double2*>(p)); }
__device__ __forceinline__ void sf_st16(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void sf_st16(double* p, double2 v) { *reinterpret_cast<double2*>(p) = v; }
template <typename T>
__device__ __forceinline__ void sf_push_planes(T* own, i64 delta, int p0, int p1, int s_base,
                                               int j0, int j1, int k0, int k1, int NJ, int NK) {
    constexpr int W = 16 / (int)sizeof(T);
    const int kv = (k1 - k0) / W, rows = j1 - j0;
    if (p1 <= p0 || kv <= 0 || rows <= 0) return;
    const i64 per_plane = (i64)rows * kv;
    const i64 total = per_plane * (p1 - p0);
    for (i64 e = threadIdx.x; e < total; e += blockDim.x) {
        const int p = p0 + (int)(e / per_plane);
        const int r = (int)(e % per_plane);
        T* src = own + (((i64)(p - s_base) * NJ + (j0 + r / kv)) * NK + (k0 + (r % kv) * W));
        sf_st16(reinterpret_cast<T*>(reinterpret_cast<char*>(src) + delta), sf_ldcg16(src));
    }
}
// ---- neighbour-only synchronisation ("pair" mode) ----
// Warp w exchanges data with warps w-1 and w+1 only, so instead of one CTA-wide barrier per streamed
// plane it meets each neighbour at a 64-thread named barrier (id w for the pair (w-1, w)).  Even warps
// meet their upper neighbour first, odd warps their lower one: all pairs (2n, 2n+1) meet concurrently,
// then all pairs (2n+1, 2n+2) -- no ripple through the CTA, and warps that are not neighbours may
// drift a step apart (the FPGA's processing elements handshake the same way, through their FIFOs).
__device__ __forceinline__ void sf_bar_pair(int id) {
    asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory");
}
template <int NW>
__device__ __forceinline__ void sf_sync_neighbours(int w) {
    if (w & 1) {
        sf_bar_pair(w);
        if (w + 1 < NW) sf_bar_pair(w + 1);
    } else {
        if (w + 1 < NW) sf_bar_pair(w + 1);
        if (w > 0) sf_bar_pair(w);
    }
}
// ---- two half-CTAs ("halves" mode) ----
// The warps of the upper and the lower half of a tile meet at their own 1-per-plane named barrier (ids 1 / 2)
// and load their own half of every input plane; only the two warps at the seam exchange rows, and they
// shake hands through producer/consumer barriers: bar.arrive (does not wait) after the step's last ring
// access, bar.sync on the other half's barrier before the next step.  The halves may therefore run up to a
// step apart -- when one is in its arithmetic the other can be in its exchange phase -- while sharing the
// tile (no halo between them, unlike two independent CTAs of half the size).
__device__ __forceinline__ void sf_bar_half(u32 upper, u32 nthreads) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %0, 0;\n\t@p bar.sync 2, %1;\n\t@!p bar.sync 1, %1;\n\t}"
                 ::"r"(upper), "r"(nthreads) : "memory");
}
template <int ID_LO, int ID_HI>
__device__ __forceinline__ void sf_seam_handshake(u32 seam_lo, u32 seam_hi) {
    // seam_lo: the last warp of the lower half, seam_hi: the first warp of the upper half (warp-uniform)
    asm volatile("{\n\t.reg .pred pa, pb;\n\tsetp.ne.u32 pa, %0, 0;\n\tsetp.ne.u32 pb, %1, 0;\n\t"
                 "@pa bar.arrive %2, 64;\n\t@pb bar.arrive %3, 64;\n\t"
                 "@pa bar.sync %3, 64;\n\t@pb bar.sync %2, 64;\n\t}"
                 ::"r"(seam_lo), "r"(seam_hi), "n"(ID_LO), "n"(ID_HI) : "memory");
}
// ---- packed float32 pairs (FADD2 / FMUL2 / FFMA2 on sm_100a) ----
__device__ __forceinline__ float2 sf_add2(float2 a, float2 b) {
    float2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(reinterpret_cast<u64&>(r))
        : "l"(reinterpret_cast<const u64&>(a)), "l"(reinterpret_cast<const u64&>(b)));
    return r;
}
__device__ __forceinline__ float2 sf_sub2(float2 a, float2 b) {
    float2 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(reinterpret_cast<u64&>(r))
        : "l"(reinterpret_cast<const u64&>(a)), "l"(reinterpret_cast<const u64&>(b)));
    return r;
}
__device__ __forceinline__ float2 sf_mul2(float2 a, float2 b) {
    float2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(reinterpret_cast<u64&>(r))
        : "l"(reinterpret_cast<const u64&>(a)), "l"(reinterpret_cast<const u64&>(b)));
    return r;
}
__device__ __forceinline__ float2 sf_fma2(float2 a, float2 b, float2 c) {
    float2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(reinterpret_cast<u64&>(r))
        : "l"(reinterpret_cast<const u64&>(a)), "l"(reinterpret_cast<const u64&>(b)),
          "l"(reinterpret_cast<const u64&>(c)));
    return r;
}
// results leave through explicit st.global (the output pointer is kept opaque to stop the compiler from
// re-deriving it per row, which would otherwise demote these to generic stores)
#ifdef SF_STG64
template <int N>
__device__ __forceinline__ void sf_stg_if(bool on, float* p, const float2 (&s)[N]) {
#pragma unroll
    for (int q = 0; q < N; ++q)
        asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %0, 0;\n\t"
                     "@q " SF_STG_V2F32 "\n\t}"
                     ::"r"((u32)on), "l"(p + 2 * q), "f"(s[q].x), "f"(s[q].y) SF_STG_HINT_ARG2 : "memory");
}
#else
template <int N>
__device__ __forceinline__ void sf_stg_if(bool on, float* p, const float2 (&s)[N]) {
#pragma unroll
    for (int q = 0; q < N; q += 2)
        asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %0, 0;\n\t"
                     "@q " SF_STG_V4F32 "\n\t}"
                     ::"r"((u32)on), "l"(p + 2 * q), "f"(s[q].x), "f"(s[q].y), "f"(s[q + 1].x), "f"(s[q + 1].y) SF_STG_HINT_ARG : "memory");
}
#endif
template <int N>
__device__ __forceinline__ void sf_stg_if(bool on, float* p, const float (&s)[N]) {
#pragma unroll
    for (int q = 0; q < N; q += 4)
        asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %0, 0;\n\t"
                     "@q " SF_STG_V4F32 "\n\t}"
                     ::"r"((u32)on), "l"(p + q), "f"(s[q]), "f"(s[q + 1]), "f"(s[q + 2]), "f"(s[q + 3]) SF_STG_HINT_ARG : "memory");
}
template <int N>
__device__ __forceinline__ void sf_stg_if(bool on, double* p, const double (&s)[N]) {
#pragma unroll
    for (int q = 0; q < N; q += 2)
        asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %0, 0;\n\t"
                     "@q " SF_STG_V2F64 "\n\t}"
                     ::"r"((u32)on), "l"(p + q), "d"(s[q]), "d"(s[q + 1]) SF_STG_HINT_ARG : "memory");
}
__device__ __forceinline__ void sf_sts_if(bool on, float* p, float v) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %0, 0;\n\t@q st.shared.f32 [%1], %2;\n\t}"
                 ::"r"((u32)on), "r"(sf_smem_addr(p)), "f"(v) : "memory");
}
__device__ __forceinline__ void sf_sts_if(bool on, double* p, double v) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %0, 0;\n\t@q st.shared.f64 [%1], %2;\n\t}"
                 ::"r"((u32)on), "r"(sf_smem_addr(p)), "d"(v) : "memory");
}
template <int V>
__device__ __forceinline__ void sf_ldp(float2* dst, const float* __restrict__ p) {
    SfVec<float, V> t = *reinterpret_cast<const SfVec<float, V>*>(p);
#pragma unroll
    for (int q = 0; q < V / 2; ++q) dst[q] = make_float2(t.v[2 * q], t.v[2 * q + 1]);
}
template <int V>
__device__ __forceinline__ void sf_stp(float* __restrict__ p, const float2* src) {
#ifdef SF_ST64
    // one 64-bit store per packed pair: a 128-bit store wants its four registers in one aligned quad, and the
    // pairs the packed arithmetic produces rarely sit in one (ptxas then copies them: 4 MOV per store)
#pragma unroll
    for (int q = 0; q < V / 2; ++q)
        asm volatile(SF_STS_V2F32 " [%0], {%1, %2};" ::"r"(sf_smem_addr(p + 2 * q)), "f"(src[q].x), "f"(src[q].y) : "memory");
#else
    SfVec<float, V> t;
#pragma unroll
    for (int q = 0; q < V / 2; ++q) { t.v[2 * q] = src[q].x; t.v[2 * q + 1] = src[q].y; }
    *reinterpret_cast<SfVec<float, V>*>(p) = t;
#endif
}
// ---- tensor memory (tcgen05, cta_group::1): one warp allocates all 512 columns for the CTA; each thread then
// moves 32-bit words between its registers and its own lane of the columns (shape 32x32b)
__device__ __forceinline__ void sf_tmem_alloc(u32* dst) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(sf_smem_addr(dst)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void sf_tmem_dealloc(u32 base) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(base) : "memory");
}
__device__ __forceinline__ void sf_tmem_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void sf_tmem_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void sf_tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void sf_tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
""" + "".join(
    '__device__ __forceinline__ void sf_tmem_st{n}(u32 a, {decl}) {{\n'
    '    asm volatile("tcgen05.st.sync.aligned.32x32b.x{n}.b32 [%0], {{{regs}}};" ::"r"(a), {ops} : "memory");\n}}\n'
    '__device__ __forceinline__ void sf_tmem_ld{n}(u32 a, {rdecl}) {{\n'
    '    asm volatile("tcgen05.ld.sync.aligned.32x32b.x{n}.b32 {{{lregs}}}, [%{n}];" : {lops} : "r"(a) : "memory");\n}}\n'.format(
        n=n, decl=", ".join("u32 v{}".format(i) for i in range(n)),
        regs=",".join("%{}".format(i + 1) for i in range(n)),
        ops=", ".join('"r"(v{})'.format(i) for i in range(n)),
        rdecl=", ".join("u32& v{}".format(i) for i in range(n)),
        lregs=",".join("%{}".format(i) for i in range(n)),
        lops=", ".join('"=r"(v{})'.format(i) for i in range(n)))
    for n in (1, 2, 4, 8, 16))


def l2_hint_defines():
    """``SFB200_L2HINT``: bit 0 = input planes are loaded with L2 evict-last priority, bit 1 = results are
    stored with evict-first priority (default: both -- measured 0.5-0.7 % on the Jacobi chains, DESIGN 3.2)."""
    bits = int(os.environ.get("SFB200_L2HINT", L2_HINT_DEFAULT))
    text = ""
    if bits & 1:
        text += "#define SF_LOAD_HINT 0x14F0000000000000ull\n"
    if bits & 2:
        text += "#define SF_STORE_HINT 0x12F0000000000000ull\n"
    st64 = int(os.environ.get("SFB200_ST64", ST64_DEFAULT))
    if st64 & 1:
        # (ptxas fuses two plain 64-bit stores back into one 128-bit store; volatile ones stay apart)
        text += "#define SF_ST64 1\n#define SF_STS_V2F32 \"{}\"\n".format(
            "st.volatile.shared.v2.f32" if st64 & 4 else "st.shared.v2.f32")
    if st64 & 2:
        text += "#define SF_STG64 1\n"
    return text


# helpers of the passes over unaligned rows (Geometry.unaligned), emitted once after STREAM_PRELUDE
UNALIGNED_PRELUDE = r"""
// ---- unaligned rows: input cells copied by cp.async into the TMA ring, results stored cell by cell ----
// one cell of a streamed input: flat element g of the field, zero when g lies outside the array (src-size 0)
template <typename T>
__device__ __forceinline__ void sf_cp_async(T* dst, const T* src, i64 g, i64 total) {
    const bool in = (unsigned long long)g < (unsigned long long)total;
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2, %3;"
                 ::"r"(sf_smem_addr(dst)), "l"(src + (in ? g : 0)), "n"((int)sizeof(T)), "r"(in ? (int)sizeof(T) : 0)
                 : "memory");
}
// the slot's mbarrier counts one arrival per copying thread, made once all of that thread's copies have landed
__device__ __forceinline__ void sf_cp_async_arrive(void* bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(sf_smem_addr(bar)) : "memory");
}
#ifdef SF_STORE_HINT
#define SF_STG_F32 "st.global.L2::cache_hint.f32 [%1], %2, %3;"
#define SF_STG_F64 "st.global.L2::cache_hint.f64 [%1], %2, %3;"
#else
#define SF_STG_F32 "st.global.f32 [%1], %2;"
#define SF_STG_F64 "st.global.f64 [%1], %2;"
#endif
// a row starts wherever (i * NJ + j) * NK puts it, so a cell is the widest store that is always aligned
__device__ __forceinline__ void sf_stg1_if(bool on, float* p, float v) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %0, 0;\n\t@q " SF_STG_F32 "\n\t}"
                 ::"r"((u32)on), "l"(p), "f"(v) SF_STG_HINT_ARG : "memory");
}
__device__ __forceinline__ void sf_stg1_if(bool on, double* p, double v) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %0, 0;\n\t@q " SF_STG_F64 "\n\t}"
                 ::"r"((u32)on), "l"(p), "d"(v) SF_STG_HINT_ARG : "memory");
}
"""

L2_HINT_DEFAULT = "3"
ST64_DEFAULT = "0"
SPLITBAR_DEFAULT = "0"
SPLITLOOP_DEFAULT = "auto"
HALO_SKIP_DEFAULT = "0"
SCHED_DEFAULT = "lpt"


class NotStreamable(Exception):
    pass


SM_COUNT = 148              # B200; the runtime overwrites it with the device's count when it initialises
EDGE_SLOWDOWN = 0.25        # how much longer a domain-edge tile may take than an interior one (boundary code)


def persistent_default(n_tiles=None, slots=None):
    """Persistent CTAs (one per SM slot, fetching work items from a list, see ``schedule_work``) pay off
    when a pass has more tiles than the device has CTA slots: whole tiles then stream without
    per-chunk warm-up planes and nothing waits for a partly filled last wave (measured: Jacobi-3D
    1024^3, 304 tiles on 148 slots, 6.5 % faster).  With fewer tiles than slots every tile is cut into
    plane ranges anyway and the plain one-CTA-per-(tile, chunk) grid is as fast or faster (hdiff: 24
    tiles, 2-D float64 chain: 137 tiles on 592 slots).  ``SFB200_PERSISTENT`` = 1 / 0 forces either."""
    env = os.environ.get("SFB200_PERSISTENT", "auto")
    if env in ("0", "1"):
        return env == "1"
    if n_tiles is None or slots is None:
        return True
    return n_tiles >= (1.0 + EDGE_SLOWDOWN) * slots


class _FieldInfo:
    def __init__(self, name, kind, dtype):
        self.name = name
        self.kind = kind              # "ext" (read from HBM) | "op" (produced in the group)
        self.dtype = dtype
        self.lag = 0                  # planes behind the stream head when produced
        self.window = 1               # planes kept in registers
        self.row_reach = 0            # max |dj| over consumers  -> rows published per side
        self.col_reach = 0            # max |dk| over consumers
        self.row_ring = 0             # exchange ring depth (0 = not published)
        self.col_ring = 0
        self.bc = None                # value consumers read outside the domain (None = never read there)
        self.copy = False             # consumers substitute the centre tap instead (``copy`` boundary)
        self.stored = False
        self.consumed = False
        self.back = 0                 # planes of history a chunk needs before its first output plane
        self.fwd = 0                  # planes beyond the last output plane of a chunk that are read
        self.need = [0, 0, 0, 0]      # halo (row lo, row hi, col lo, col hi) this field must be valid on


class GroupAnalysis:
    """Lags, windows, rings and halos of a fusion group (see the module docstring)."""

    def __init__(self, program: StencilProgram, ops: List[StencilOp], exchange_cols: bool):
        self.program = program
        self.ops = ops
        self.ndim = len(program.shape)
        if self.ndim not in (2, 3):
            raise NotStreamable("only 2-D and 3-D programs stream")
        self.exchange_cols = exchange_cols
        self.dtype = ops[0].data_type
        if self.dtype not in (dtypes.float32, dtypes.float64):
            raise NotStreamable("only float32/float64 fields stream")
        self.fields: Dict[str, _FieldInfo] = collections.OrderedDict()
        self.taps: Dict[str, List[Tuple[str, int, int, int]]] = {}
        # lower-dimensional array inputs (``input_dims`` a strict subset of the iterators,
        # ``kernel_chain_graph.py:382-389``): not streamed -- read straight from global memory
        # (L1/L2-resident), once per kernel when they do not vary along the streamed dimension
        self.aux = collections.OrderedDict()                 # name -> Field
        self.aux_taps: Dict[str, List[Tuple[str, tuple]]] = {}
        self.aux_reach: Dict[str, List[int]] = {}            # name -> [back, fwd] along the streamed dim
        self.aux_bc: Dict[str, float] = {}
        self.copy_taps = set()                               # (operator, field) read with a ``copy`` boundary
        self.copy_reach = {}                                 # copy_taps -> (min, max) offset along the streamed dim
        produced = {op.name for op in ops}
        # fields of the group that operators outside it read: they have to be written to HBM
        later = set()
        for op in program.ops:
            if op not in ops:
                later.update(f for f in op.accesses if f in produced)
        for op in ops:
            if op.data_type != self.dtype:
                raise NotStreamable("mixed result types in group")
            taps = []
            for field in op.accesses:
                f = program.fields[field]
                if f.data_type != self.dtype:
                    raise NotStreamable("field {} has a different type".format(field))
                if list(f.dims) != list(program.iterators):
                    bc = op.boundary_conditions.get(field)
                    if f.kind != "input" or (bc is not None and bc["btype"] == "copy"):
                        raise NotStreamable("lower-dimensional field {} cannot be read directly".format(field))
                    self.aux[field] = f
                    self.aux_taps.setdefault(op.name, []).extend((field, off) for off in op.offsets3(field))
                    if bc is not None:
                        val = float(bc["value"]) if bc["btype"] == "constant" else float(JUNK_VAL)
                        if self.aux_bc.setdefault(field, val) != val:
                            raise NotStreamable("consumers of {} disagree on the boundary value".format(field))
                    continue
                if field not in self.fields:
                    if field in produced:
                        raise NotStreamable("operators out of order")
                    self.fields[field] = _FieldInfo(field, "ext", f.data_type)
                for off in op.offsets3(field):
                    if self.ndim == 3:
                        d, dj, dk = off
                    else:
                        d, dj, dk = off[1], 0, off[2]
                    taps.append((field, d, dj, dk))
                bc = op.boundary_conditions.get(field)
                if any((t[1], t[2], t[3]) != (0, 0, 0) for t in taps if t[0] == field):
                    if bc is None:
                        raise NotStreamable("missing boundary condition")
                    info = self.fields[field]
                    if bc["btype"] == "copy":
                        # an out-of-domain tap reads the field's centre tap at the consumer's own cell
                        # (``intel_fpga.py:179-185,225-227``): decided where the tap is *consumed*, so the
                        # centre plane has to be in the window and nothing is fixed where the field is produced
                        if info.bc is not None:
                            raise NotStreamable("consumers of {} disagree on the boundary handling".format(field))
                        info.copy = True
                        self.copy_taps.add((op.name, field))
                        ds = [t[1] for t in taps if t[0] == field]
                        self.copy_reach[(op.name, field)] = (min(ds + [0]), max(ds + [0]))
                        if (field, 0, 0, 0) not in taps:
                            taps.append((field, 0, 0, 0))
                    else:
                        val = float(bc["value"]) if bc["btype"] == "constant" else float(JUNK_VAL)
                        if info.copy or (info.bc is not None and info.bc != val):
                            raise NotStreamable("consumers of {} disagree on the boundary value".format(field))
                        info.bc = val
            self.taps[op.name] = taps
            info = _FieldInfo(op.name, "op", op.data_type)
            info.stored = (program.fields[op.name].kind == "output") or (op.name in later)
            self.fields[op.name] = info
        for op in ops:
            for (field, d, dj, dk) in self.taps[op.name]:
                self.fields[field].consumed = True
        for op in ops:
            info = self.fields[op.name]
            if not info.stored and not info.consumed:
                raise NotStreamable("dead operator {}".format(op.name))
        if not any(i.kind == "ext" for i in self.fields.values()):
            raise NotStreamable("group reads no full-dimensional field")
        self._lags()
        self.tmem_ages = self._tmem_slots()
        self._halos()
        spos = 3 - self.ndim                      # position of the streamed iterator in (i, j, k)
        for op in ops:
            for (field, off) in self.aux_taps.get(op.name, []):
                if off[spos] is not None:
                    r = self.aux_reach.setdefault(field, [0, 0])
                    r[0] = max(r[0], self.fields[op.name].back + max(0, -off[spos]))
                    r[1] = max(r[1], self.fields[op.name].fwd + max(0, off[spos]))

    def aux_split(self, off):
        """(d_stream, d_row, d_col) of a lower-dimensional tap, None for dimensions the field lacks."""
        if self.ndim == 3:
            return off[0], off[1], off[2]
        return off[1], None, off[2]

    def aux_hoisted(self):
        """Distinct (field, offsets) taps that do not vary along the streamed dimension."""
        out = []
        for op in self.ops:
            for (field, off) in self.aux_taps.get(op.name, []):
                if self.aux_split(off)[0] is None and (field, off) not in out:
                    out.append((field, off))
        return out

    def _is_exchange(self, dj, dk):
        return dj != 0 or (self.exchange_cols and dk != 0)

    def _lags(self):
        f = self.fields
        for op in self.ops:
            lag = 0
            for (field, d, dj, dk) in self.taps[op.name]:
                lag = max(lag, f[field].lag + d + (1 if self._is_exchange(dj, dk) else 0), f[field].lag)
            f[op.name].lag = lag
        # delay the loading of inputs that are only needed late (keeps their windows short)
        for name, info in f.items():
            if info.kind != "ext":
                continue
            slack = None
            for op in self.ops:
                for (field, d, dj, dk) in self.taps[op.name]:
                    if field == name:
                        s = f[op.name].lag - d - (1 if self._is_exchange(dj, dk) else 0)
                        slack = s if slack is None else min(slack, s)
            info.lag = max(0, slack or 0)
        for op in self.ops:
            for (field, d, dj, dk) in self.taps[op.name]:
                src = f[field]
                age = f[op.name].lag - d - src.lag
                assert age >= 0
                src.window = max(src.window, age + 1)
                src.row_reach = max(src.row_reach, abs(dj))
                src.col_reach = max(src.col_reach, abs(dk))
                if dj != 0:
                    assert age >= 1
                    src.row_ring = max(src.row_ring, age + 1)
                if self.exchange_cols and dk != 0:
                    assert age >= 1
                    src.col_ring = max(src.col_ring, age + 1)
        # history needed before the first output plane of a chunk
        for op in reversed(self.ops):
            for (field, d, dj, dk) in self.taps[op.name]:
                f[field].back = max(f[field].back, f[op.name].back + max(0, -d))
                f[field].fwd = max(f[field].fwd, f[op.name].fwd + max(0, d))

    def _tmem_slots(self):
        """{field: age} of the window slots that may wait in tensor memory between two uses.  The oldest plane of
        a window (age window - 1) qualifies when every read of it at that age is an own-cell tap (dj == dk == 0):
        no shuffle and no exchange ring reads it, only the thread that holds it.  Its owner parks it after its
        last use one step younger and fetches it back a step later, so its registers are free in between."""
        f = self.fields
        out = collections.OrderedDict()
        for name, info in f.items():
            age = info.window - 1
            if not info.consumed or age < 1:
                continue
            reads = [(dj, dk) for op in self.ops for (field, d, dj, dk) in self.taps[op.name]
                     if field == name and f[op.name].lag - d - info.lag == age]
            if reads and all(dj == 0 and dk == 0 for (dj, dk) in reads):
                out[name] = age
        return out

    def _halos(self):
        f = self.fields
        for op in reversed(self.ops):
            need = f[op.name].need
            for (field, d, dj, dk) in self.taps[op.name]:
                n = f[field].need
                n[0] = max(n[0], need[0] + max(0, -dj))
                n[1] = max(n[1], need[1] + max(0, dj))
                n[2] = max(n[2], need[2] + max(0, -dk))
                n[3] = max(n[3], need[3] + max(0, dk))
        ext = [i for i in f.values() if i.kind == "ext"]
        self.halo = [max(i.need[s] for i in ext) for s in range(4)]

    @property
    def ext_fields(self):
        return [i for i in self.fields.values() if i.kind == "ext"]

    @property
    def max_lag(self):
        return max(i.lag for i in self.fields.values())

    def t_begin_offset(self):
        """first step = chunk_begin + this (<= 0)"""
        return min(-i.back + i.lag for i in self.fields.values())

    def t_end_offset(self):
        """last step + 1 = chunk_end + this"""
        return max(i.lag for i in self.fields.values() if i.stored)

    def window_registers(self, R, V):
        per = self.dtype.bytes // 4
        return sum(i.window for i in self.fields.values() if i.consumed) * R * V * per

    def register_estimate(self, R, V, tmem=False):
        """Registers per thread the generated kernel needs: the planes of every window that are
        live across steps (the oldest plane of a window dies while the newest is being produced)
        plus what is in flight -- the plane being produced, its consumer's result, the pre-fetched
        neighbour cells of the next operator, addresses, masks and loop state.  The constant part is
        fitted to ptxas' allocations of the Jacobi/hdiff kernels (spill-free iff estimate <= limit).
        ``tmem``: the slots of ``tmem_ages`` wait in tensor memory, not in registers, across a step."""
        per = self.dtype.bytes // 4
        live = sum(max(1, i.window - 1) for i in self.fields.values() if i.consumed)
        if tmem:
            live -= len(self.tmem_ages)
        hoisted = 0
        for (field, off) in self.aux_hoisted():
            _, dr, dc = self.aux_split(off)
            hoisted += (R if dr is not None else 1) * (V if dc is not None else 1) * per
        per_step = 0                  # taps loaded per plane: live only while their operator is evaluated
        for op in self.ops:
            n = 0
            for (field, off) in self.aux_taps.get(op.name, []):
                ds, dr, dc = self.aux_split(off)
                if ds is not None:
                    n += (R if dr is not None else 1) * (V if dc is not None else 1) * per
            per_step = max(per_step, n)
        hoisted += per_step
        return (live + 2) * R * V * per + 8 + min(10, R * V * per) * len(self.ops) + hoisted


class Geometry:
    def __init__(self, ana: GroupAnalysis, V, R, WR, WC, prefetch, KS=32, sync="cta", direct=False, tmem=False,
                 unaligned=False):
        """``KS`` = threads per tile row.  32 (a warp per row, k-neighbours by shuffle) in general;
        for groups without k-taps on a narrow innermost dimension the whole extent is one row of
        ``KS = NK / V`` threads and thread t owns row group t / KS ("flat lanes": no idle lanes).
        ``unaligned``: the innermost rows are not a multiple of 16 bytes long, which a tiled TMA map of 2 or 3
        dimensions needs for its strides.  The threads then copy the cells of the input planes themselves
        (``cp.async``, see StreamKernelGen._emit_copy_issue) into the same shared-memory layout."""
        self.V, self.R, self.WR, self.WC, self.KS = V, R, WR, WC, KS
        self.unaligned = bool(unaligned)
        self.NT = KS * WR * WC
        ktaps = any(i.col_reach for i in ana.fields.values())
        if KS != 32 and (WC != 1 or self.NT % 32 or (ktaps and KS not in (8, 16))):
            raise NotStreamable("narrow rows need a single column tile (and a power-of-two width for k-taps)")
        if self.NT > 1024:
            raise NotStreamable("too many threads")
        self.TR, self.TC = WR * R, WC * KS * V
        h = ana.halo
        self.HJ0, self.HJ1 = h[0], h[1]
        self.HK0 = -(-h[2] // V) * V
        self.HK1 = -(-h[3] // V) * V
        self.BJ = self.TR - self.HJ0 - self.HJ1
        self.BK = self.TC - self.HK0 - self.HK1
        self.P = prefetch
        # "direct" rows: a thread reads the j-neighbour rows of a streamed input straight from the
        # plane TMA put into shared memory (any thread may read any row of it) instead of from an
        # exchange ring the owners re-publish them into -- two shared-memory stores per thread and
        # plane less.  The TMA ring then keeps a plane as long as its rows are read (``keep`` extra
        # slots).  Only for inputs whose out-of-domain cells need no fix-up (TMA's zero fill is the
        # boundary value), 3-D tiles, CTA-wide synchronisation.
        self.direct = {}
        # (not with unaligned rows: the copies fill the cells outside a row with the neighbouring rows' data, and
        # only the registers get the boundary value)
        if direct and ana.ndim == 3 and sync != "pair" and not self.unaligned:
            for i in ana.ext_fields:
                if i.row_ring and not i.col_ring and (i.bc is None or float(i.bc) == 0.0):
                    self.direct[i.name] = i.row_ring - 1
        self.keep = max(self.direct.values()) if self.direct else 0
        self.D = prefetch + 1 + self.keep
        if ana.ndim == 2:
            self.BJ = 1
        if self.BJ < 1 or self.BK < V:
            raise NotStreamable("tile smaller than its halo")
        for i in ana.fields.values():
            if i.row_reach > R:
                raise NotStreamable("row reach exceeds rows per thread")
            if i.col_reach > V:
                raise NotStreamable("column reach exceeds the vector width")
        if self.TR > 256:
            raise NotStreamable("tile taller than a TMA box")
        self.box_cols = min(self.TC, 256)
        if self.TC % self.box_cols:
            raise NotStreamable("tile width not a multiple of the TMA box")
        # "pair" synchronisation: every warp loads its own part of each input plane (own TMA box, own
        # mbarriers) and meets only its two neighbours once per plane.  Needs whole row groups per
        # warp (3-D, one column of warps) or one row of warps (2-D), and one named barrier per pair.
        nw = self.NT // 32
        self.NW = nw
        # "flags" synchronisation: no CTA-wide barrier in the streamed loop; every published field has an
        # mbarrier its producers arrive on and its consumers wait for a step later (StreamKernelGen.flags)
        self.flags = (sync == "flags")
        self.pair = False
        if sync == "pair" and 2 <= nw <= 16:
            if ana.ndim == 3 and WC == 1 and 32 % KS == 0 and self.TC <= 256:
                self.pair = True
                self.warp_rows = (32 // KS) * R
                self.box = [self.TC, self.warp_rows, 1]
            elif ana.ndim == 2 and WR == 1 and KS == 32 and 32 * V <= 256:
                self.pair = True
                self.warp_rows = 1
                self.box = [32 * V, 1]
        if not self.pair:
            self.box = [self.box_cols, self.TR, 1] if ana.ndim == 3 else [self.box_cols, 1]
        # "halves": two half-CTAs sharing a tile (see sf_bar_half in the prelude)
        self.halves = bool(sync == "halves" and ana.ndim == 3 and WC == 1 and not self.direct and nw % 2 == 0
                           and WR % 2 == 0 and self.TC == self.box_cols and (WR // 2) % max(1, 32 // KS) == 0)
        if self.halves:
            self.box = [self.box_cols, self.TR // 2, 1]
        self.smem = self._smem(ana)
        # tensor memory: the window slots of ``ana.tmem_ages`` wait there between two uses (StreamKernelGen).  The
        # CTA allocates all 512 columns, so it must be alone on its SM; warp w reaches TMEM lanes 32 (w % 4) ...
        # + 31 and owns 128 columns of them (at most 16 warps), two planes per slot, each padded to a power of two
        self.tmem_cols = 0
        if tmem and ana.ndim == 3 and ana.tmem_ages and nw <= 16:
            words = R * V * ana.dtype.bytes // 4
            self.tmem_cols = 1 << (words - 1).bit_length()
            if 2 * self.tmem_cols * len(ana.tmem_ages) > 128:
                self.tmem_cols = 0
        self.tmem = bool(self.tmem_cols)
        if self.tmem:
            self.tmem_off = self.smem          # the address tcgen05.alloc returns
            self.smem += 16
            if resident_estimate(self) != 1:
                self.tmem, self.tmem_cols, self.smem = False, 0, self.tmem_off

    def _smem(self, ana):
        b = ana.dtype.bytes
        off = 0
        self.tile_off, self.xrow_off, self.xcol_off = {}, {}, {}
        for i in ana.ext_fields:
            self.tile_off[i.name] = off
            off += self.D * self.TR * self.TC * b
            off = (off + 127) & ~127
        for i in ana.fields.values():
            if i.row_ring and i.name not in self.direct:
                self.xrow_off[i.name] = off
                off += i.row_ring * self.WR * 2 * i.row_reach * self.TC * b
                off = (off + 127) & ~127
            if i.col_ring:
                self.xcol_off[i.name] = off
                off += i.col_ring * self.WR * self.WC * 2 * self.R * i.col_reach * b
                off = (off + 127) & ~127
        self.bar_off = off
        off += 8 * self.D * (self.NW if self.pair else (2 if self.halves else 1))
        self.item_off = off            # persistent CTAs: the work item thread 0 fetched for everybody
        off += 16
        self.sbar_off = off            # split CTA barrier (see StreamKernelGen.split_barrier)
        off += 16
        self.fbar_off = off            # one mbarrier per published field ("flags" synchronisation)
        off += (8 * len(ana.fields) + 15) & ~15
        return off


def _fmt_off(x):
    return str(x).replace("-", "m")


class StreamKernelGen:
    """Emits the CUDA C++ of one fused pass.

    Two code-shape decisions matter for the instruction count (the pass is issue-bound once it is
    fused, see DESIGN.md section 3.2):

    * the streamed loop is unrolled ``U`` times, ``U`` a common multiple of the periods of the rotating
      resources (register windows, TMA ring, exchange rings), so that every window slot and ring slot
      is a compile-time constant: no register-to-register window rotation, no modulo arithmetic;
    * float32 groups compute on *pairs* of neighbouring cells with Blackwell's packed
      ``add/mul/fma.rn.f32x2`` (SASS ``FADD2/FMUL2/FFMA2``): one issue slot per two cells.  Taps whose
      two cells do not sit in one aligned register pair (odd k-offsets, cells from another lane) fall
      back to two scalar operations, which still write an aligned pair.
    """

    def __init__(self, program: StencilProgram, ops: List[StencilOp], ana: GroupAnalysis, geo: Geometry,
                 specialize=None, max_unroll=None, pack=None, persistent=None, peer_push=False):
        self.program, self.ops, self.ana, self.geo = program, ops, ana, geo
        self.specialize = specialize or {}
        self.ct = ana.dtype
        self.T = ctype_of(self.ct)
        self.NI, self.NJ, self.NK = program.shape3
        self.NS = program.shape[0]                     # extent of the streamed dimension
        self.scalars = []
        for op in ops:
            for s in op.scalars:
                if s not in program.constants and s not in self.specialize and s not in self.scalars:
                    self.scalars.append(s)
        self.lines: List[str] = []
        if pack is None:
            pack = os.environ.get("SFB200_PACK", "1") != "0"
        if max_unroll is None:
            max_unroll = int(os.environ.get("SFB200_UNROLL", "6"))
        self.G = 2 if (pack and self.ct == dtypes.float32 and geo.V % 2 == 0) else 1
        self.VH = geo.V // self.G
        self.ET = "float2" if self.G == 2 else self.T
        self.U = self._choose_unroll(max(1, max_unroll))
        self.pipeline = os.environ.get("SFB200_PIPELINE", "1") != "0"
        self.fast_path = os.environ.get("SFB200_FASTPATH", "1") != "0"
        # separate loops for the trips with and without boundary code (see generate): measured +1.4 % on the
        # float64 2-D chain; the 3-D Jacobi pass sits at its register limit and spills with it (-19 %)
        split = os.environ.get("SFB200_SPLITLOOP", SPLITLOOP_DEFAULT)
        self.split_loop = (ana.ndim == 2) if split == "auto" else split != "0"
        self.with_bc = True
        self._tmp = 0
        # split CTA barrier: instead of one __syncthreads at the end of a streamed step every warp *arrives*
        # (one elected lane, after a __syncwarp) on an mbarrier as soon as it has published its last edge rows
        # and read its last neighbour rows of the step, and *waits* at the end of the step -- what lies in
        # between (the arithmetic and the stores of the group's last operator, which nobody in the CTA reads)
        # overlaps with the slower warps catching up
        self.split_barrier = (os.environ.get("SFB200_SPLITBAR", SPLITBAR_DEFAULT) != "0") and not geo.pair
        # "flags" synchronisation (Geometry.flags): the CTA-wide barrier at the end of every streamed step is
        # replaced by one mbarrier per published field.  A warp arrives on it right after it has stored its
        # edge rows / columns of the field's new plane and waits for it a step later, just before it reads its
        # neighbours' -- so warps may run up to a step apart, and the shared-memory, shuffle and arithmetic
        # phases of different warps overlap instead of all warps hitting the same pipe at the same time (the
        # FPGA design's processing elements are coupled the same way: through their FIFOs, not by a global
        # clock-enable).  Needs every exchange ring to be read, in program order, before it is written again
        # (see _flags_ok); anything else keeps the barrier.
        self.fbar = {}
        self.flags = bool(geo.flags and not geo.pair and self.pipeline and self.U % 2 == 0 and self._flags_ok())
        if getattr(geo, "halves", False):
            if self.U % 2:
                raise NotStreamable("half-CTA synchronisation needs an even unroll factor")
            self.split_barrier = False
        if self.flags:
            self.split_barrier = False
        self._waited = set()
        # tensor memory (Geometry.tmem): the two planes of a slot in flight alternate between two column sets, so
        # the unrolled loop needs an even number of steps and static window slots
        self.tmem = bool(geo.tmem and self.U % 2 == 0 and all(self.wperiod(ana.fields[n]) for n in ana.tmem_ages))
        self._tm_loaded, self._tm_waited = set(), set()
        self.rotate_rows, self.skip_warps, self.skip_from = self._halo_warps()
        self.ops_limit = len(ops)
        # how produced planes get their out-of-domain cells set to the boundary value (see _finish_field)
        self.bc_mode = os.environ.get("SFB200_BC_MODE", "auto")
        # persistent scheduling (see schedule_work): tiles of the in-plane grid
        # slab mode: the kernel stores the edge planes of its results a second time, straight into the
        # neighbouring GPUs' halo planes (peer stores over NVLink), instead of leaving them to a copy
        self.peer_push = bool(peer_push)
        gx = -(-self.NK // geo.BK)
        gy = -(-self.NJ // geo.BJ) if ana.ndim == 3 else 1
        self.n_tiles = gx * gy
        if persistent is None:
            persistent = persistent_default(self.n_tiles, SM_COUNT * resident_estimate(geo))
        self.persistent = bool(persistent)
        if self.bc_mode not in ("thread", "cta"):
            # per-thread fix-ups (only warps that own out-of-domain cells enter the code) paid off while
            # domain-edge tiles could hold up the work list (halving rounds: Jacobi-3D 1024^3 4.17 -> 4.05 ms).
            # With the longest-first list the edge tiles stream first and the plain per-CTA test -- branch-free,
            # fewer registers (hdiff: 123 instead of 128 and no spill, 0.163 vs 0.180 ms) -- is the faster one
            # again (3.79 -> 3.73 ms, profiles/r02_sweep_sync_config1.txt)
            sched = os.environ.get("SFB200_SCHED", SCHED_DEFAULT)
            self.bc_mode = "thread" if (self.persistent and sched not in ("lpt", "rows")) else "cta"

    def _published(self, info):
        return bool((info.row_ring and info.name not in self.geo.direct) or info.col_ring)

    def _flags_ok(self):
        """Flag synchronisation is safe when, for every published field, (1) its ring is two deep and read at
        age 1 only, (2) its only reader through the ring is the operator right after its producer, whose
        neighbour data is gathered *before* the producer's new plane is published (software pipelining), so
        that a warp's arrival for step t also says "my reads of step t-1's slot are done"; (3) every streamed
        input is published (its arrival doubles as "tile slot read" for the TMA ring)."""
        a = self.ana
        names = [op.name for op in self.ops]
        for info in a.fields.values():
            if info.kind == "ext" and not self._published(info):
                return False
            if not self._published(info):
                continue
            if info.row_ring not in (0, 2) or info.col_ring not in (0, 2):
                return False
            readers = []
            for op in self.ops:
                for (field, d, dj, dk) in a.taps[op.name]:
                    if field == info.name and a._is_exchange(dj, dk) and op.name not in readers:
                        readers.append(op.name)
            expect = 0 if info.kind == "ext" else names.index(info.name) + 1
            if expect >= len(names) or readers != [names[expect]]:
                return False
            if not self._can_gather_early(self.ops[expect]):
                return False
            self.fbar[info.name] = len(self.fbar)
        return bool(self.fbar)

    def _flag_wait(self, info, age, u, indent=2):
        """Before the first read of what other warps published of ``info`` at step (t - age)."""
        if not self.flags or info.name not in self.fbar or (info.name, age) in self._waited:
            return
        self._waited.add((info.name, age))
        self.emit("sf_mbar_wait(&fbars[{}], {}u);".format(self.fbar[info.name], (u - age) % 2), indent)

    def _flag_arrive(self, info):
        if self.flags and info.name in self.fbar:
            self.emit("__syncwarp(); if (sf_elect_one()) sf_mbar_arrive(&fbars[{}]);".format(self.fbar[info.name]), 2)

    # ------------------------------------------------------------------ unrolling
    def _choose_unroll(self, cap):
        a, g = self.ana, self.geo
        windows = [i.window for i in a.fields.values() if i.consumed and i.window > 1]
        rings = [i.row_ring for i in a.fields.values() if i.row_ring and i.name not in g.direct]
        rings += [i.col_ring for i in a.fields.values() if i.col_ring]
        wmax = max(windows + [1])
        for periods in ([g.D] + rings, [g.D], []):
            base = 1
            for n in periods:
                base = base * n // math.gcd(base, n)
            u = base * -(-wmax // base)          # smallest multiple of the smem periods covering every window
            u *= max(1, int(os.environ.get("SFB200_UNROLL_MULT", "1")))   # (experiment: amortise the trip-end copies)
            if u <= cap:
                return u
        return 1

    def static(self, period):
        return self.U % period == 0

    def wperiod(self, info):
        """Renaming period of a register window.  Slots that hold no live plane cost no register, so
        a window is padded to the unroll factor whenever that is large enough; only a window longer
        than the unroll factor falls back to rotation by moves (period 0)."""
        if info.window == 1:
            return 1
        if self.U >= info.window:
            return self.U
        return info.window if self.U % info.window == 0 else 0

    def wslot(self, info, age, u):
        """window slot holding the plane of ``age`` once the field has been produced at position u"""
        n = self.wperiod(info)
        if n == 1:
            return 0
        if n:
            return (u - age) % n
        return age

    def ring_slot(self, var, n, age, u):
        if self.static(n):
            return str((u - age) % n)
        if age == 0:
            return var
        return "(({rv} + {k}) % {n})".format(rv=var, k=n - (age % n), n=n)

    # ------------------------------------------------------------------ small emit helpers
    def emit(self, text, indent=1):
        self.lines.append("  " * indent + text)

    def lit(self, v):
        return literal(v, self.ct)

    def tmp(self):
        self._tmp += 1
        return "q{}".format(self._tmp)

    def cellref(self, vec, c):
        if self.G == 2:
            return "{}[{}].{}".format(vec, c // 2, "xy"[c % 2])
        return "{}[{}]".format(vec, c)

    def ldv(self, dst, src):
        if self.G == 2:
            return "sf_ldp<{}>({}, {});".format(self.geo.V, dst, src)
        return "sf_ldv<{}, {}>({}, {});".format(self.T, self.geo.V, dst, src)

    def stv(self, dst, src):
        if self.G == 2:
            return "sf_stp<{}>({}, {});".format(self.geo.V, dst, src)
        return "sf_stv<{}, {}>({}, {});".format(self.T, self.geo.V, dst, src)

    # ------------------------------------------------------------------ kernel text
    def generate(self):
        g, a = self.geo, self.ana
        T, V, R = self.T, g.V, g.R
        e = self.emit
        ndim = a.ndim
        ext = a.ext_fields
        U = self.U
        stored = [i for i in a.fields.values() if i.stored]
        if g.unaligned:
            params = ["const {}* __restrict__ in_{}".format(T, n) for n in range(len(ext))]
        else:
            params = ["const __grid_constant__ CUtensorMap tm_{}".format(n) for n in range(len(ext))]
        params += ["{}* __restrict__ o_{}".format(T, n) for n in range(len(stored))]
        self.aux_name = {name: "x_{}".format(n) for n, name in enumerate(a.aux)}
        params += ["const {}* __restrict__ {}".format(T, self.aux_name[name]) for name in a.aux]
        self.sc_name = {s: "s{}".format(n) for n, s in enumerate(self.scalars)}
        params += ["const {} {}".format(ctype_of(self.program.fields[s].data_type), self.sc_name[s])
                   for s in self.scalars]
        params += ["const int s_base", "const int s_begin", "const int s_end"]
        params += ["int* __restrict__ work_tab"] if self.persistent else ["const int chunk"]
        if self.peer_push:
            # per stored field: byte distance from a cell of this rank's buffer to the same cell of the
            # lower / upper neighbour's buffer, and the planes that go there (< lo_end, >= hi_begin)
            for n in range(len(stored)):
                params += ["const i64 pd_lo_{}".format(n), "const i64 pd_hi_{}".format(n),
                           "const int pe_lo_{}".format(n), "const int pb_hi_{}".format(n)]
        self.fid = {name: "f{}".format(n) for n, name in enumerate(a.fields)}
        static_d = self.static(g.D)
        if g.direct and not static_d:
            raise NotStreamable("direct input rows need a TMA ring whose depth divides the unroll factor")

        # ---- once per CTA: thread coordinates, shared memory, barriers, register windows
        e("extern __shared__ __align__(1024) unsigned char sf_smem[];")
        if g.KS == 32:
            e("const int lane = threadIdx.x & 31;")
            e("const int warp = threadIdx.x >> 5;")
        else:
            e("const int lane = threadIdx.x % {};          // column slot within the row".format(g.KS))
            e("const int warp = threadIdx.x / {};          // row group".format(g.KS))
        if self.rotate_rows:
            e("const int wr = (warp + {}) % {};        // row groups dealt to the warps rotated by one (see _halo_warps)".format(g.WR - 1, g.WR))
        else:
            e("const int wr = warp / {};".format(g.WC))
        e("const int wc = warp % {};".format(g.WC))
        e("(void)wr; (void)wc;")
        e("const int c0 = (wc * {} + lane) * {};            // first owned column inside the tile".format(g.KS, V))
        if ndim == 3:
            e("const int r0 = wr * {};".format(R))
        for n, i in enumerate(ext):
            e("{T}* const tile_{f} = reinterpret_cast<{T}*>(sf_smem + {o});".format(
                T=T, f=self.fid[i.name], o=g.tile_off[i.name]))
        for i in a.fields.values():
            if i.row_ring and i.name not in g.direct:
                e("{T}* const xrow_{f} = reinterpret_cast<{T}*>(sf_smem + {o});".format(
                    T=T, f=self.fid[i.name], o=g.xrow_off[i.name]))
            if i.col_ring:
                e("{T}* const xcol_{f} = reinterpret_cast<{T}*>(sf_smem + {o});".format(
                    T=T, f=self.fid[i.name], o=g.xcol_off[i.name]))
        e("unsigned long long* const bars = reinterpret_cast<unsigned long long*>(sf_smem + {});".format(g.bar_off))
        e("if (threadIdx.x == 0) {")
        e("for (int s = 0; s < {}; ++s) sf_mbar_init(&bars[s], {});".format(
            g.D * (g.NW if g.pair else (2 if g.halves else 1)), self._copy_threads()[0] if g.unaligned else 1), 2)
        if self.split_barrier:
            e("sf_mbar_init(sf_smem + {}, {});".format(g.sbar_off, g.NT // 32), 2)
        for n in range(len(self.fbar) if self.flags else 0):
            e("sf_mbar_init(sf_smem + {}, {});".format(g.fbar_off + 8 * n, g.NT // 32), 2)
        e("sf_fence_barrier_init();", 2)
        e("}")
        e("__syncthreads();")
        zero = "make_float2(0.0f, 0.0f)" if self.G == 2 else self.lit(0)
        for i in a.fields.values():
            if i.consumed:
                W = self.wperiod(i) or i.window
                e("{ET} w_{f}[{W}][{R}][{VH}];".format(ET=self.ET, f=self.fid[i.name], W=W, R=R, VH=self.VH))
                e("#pragma unroll")
                e("for (int a = 0; a < {}; ++a)".format(W))
                e("#pragma unroll", 2)
                e("for (int r = 0; r < {}; ++r)".format(R), 2)
                e("#pragma unroll", 3)
                e("for (int v = 0; v < {}; ++v) w_{}[a][r][v] = {};".format(self.VH, self.fid[i.name], zero), 3)
            if i.row_ring and i.name not in g.direct and not self.static(i.row_ring):
                e("int xr_{} = 0;".format(self.fid[i.name]))
            if i.col_ring and not self.static(i.col_ring):
                e("int xc_{} = 0;".format(self.fid[i.name]))
        if static_d:
            e("u32 phase = 0;")
        else:
            e("int slot = 0; u32 phase = 0;")
        e("const int warp_u = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);   // warp-uniform")
        if self.skip_from < len(self.ops):
            e("const bool halo_warp = {};".format(" || ".join("warp_u == {}".format(w) for w in self.skip_warps)))
        if self.flags:
            e("unsigned long long* const fbars = reinterpret_cast<unsigned long long*>(sf_smem + {});".format(g.fbar_off))
        if self.split_barrier:
            e("unsigned long long* const sbar = reinterpret_cast<unsigned long long*>(sf_smem + {});".format(g.sbar_off))
            if U % 2:
                e("u32 sphase = 0;")
        if self.tmem:
            e("u32* const sf_tmem = reinterpret_cast<u32*>(sf_smem + {});".format(g.tmem_off))
            if self.persistent:
                self._emit_tmem_alloc()

        # ---- the segment(s) this CTA streams: a tile and a range of planes of the streamed dimension
        gx = -(-self.NK // g.BK)
        if self.persistent:
            # persistent CTAs (one per SM slot) fetch work items -- (tile, first plane, end plane),
            # planes relative to s_begin -- from the list the host scheduled (``schedule_work``): item
            # blockIdx.x first, then whatever is next on the shared counter.  Items are ordered so
            # that CTAs running at the same time hold adjacent tiles at the same planes; fetching
            # dynamically lets CTAs on cheap (interior) tiles take over work from those on domain-edge
            # tiles, which run the boundary code in every step.
            e("int* const sf_item = reinterpret_cast<int*>(sf_smem + {});".format(g.item_off))
            e("int item = blockIdx.x;")
            e("#pragma unroll 1")
            e("while (item < __ldg(work_tab + 2)) {")
            e("const int tile = work_tab[3 + 3 * item];")
            e("const int p_begin = work_tab[4 + 3 * item];")
            e("const int p_end = work_tab[5 + 3 * item];")
            e("const int tile_k0 = (tile % {}) * {};".format(gx, g.BK))
            if ndim == 3:
                e("const int tile_j0 = (tile / {}) * {};".format(gx, g.BJ))
            e("const int c_begin = s_begin + p_begin;")
            e("const int c_end = s_begin + p_end;")
        else:
            e("{")
            e("const int tile_k0 = blockIdx.x * {};".format(g.BK))
            if ndim == 3:
                e("const int tile_j0 = blockIdx.y * {};".format(g.BJ))
            e("const int c_begin = s_begin + blockIdx.z * chunk;")
            e("const int c_end = min(c_begin + chunk, s_end);")
            e("if (c_begin >= c_end) return;")
            if self.tmem:
                self._emit_tmem_alloc()
        e("const int gk = tile_k0 - {} + c0;                 // global k of the first owned column".format(g.HK0))
        if ndim == 3:
            e("const int gj0 = tile_j0 - {} + r0;".format(g.HJ0))
        # in-domain mask of the owned cells, store mask of the owned rows
        e("u32 cmask = 0;")
        e("u32 smask = 0;")
        if g.unaligned:
            e("u32 stmask = 0;")
        e("#pragma unroll")
        e("for (int r = 0; r < {}; ++r) {{".format(R))
        if ndim == 3:
            e("const bool rin = (gj0 + r) >= 0 && (gj0 + r) < {};".format(self.NJ), 2)
            e("const bool rst = rin && (r0 + r) >= {} && (r0 + r) < {};".format(g.HJ0, g.TR - g.HJ1), 2)
        else:
            e("const bool rin = true, rst = true;", 2)
        e("#pragma unroll", 2)
        e("for (int v = 0; v < {}; ++v)".format(V), 2)
        e("if (rin && (gk + v) >= 0 && (gk + v) < {}) cmask |= 1u << (r * {} + v);".format(self.NK, V), 3)
        e("if (rst && c0 >= {} && c0 < {} && gk < {}) smask |= 1u << r;".format(g.HK0, g.TC - g.HK1, self.NK), 2)
        if g.unaligned:
            # store mask of the owned cells: the last vector of a row is ragged
            e("if ((smask >> r) & 1u) stmask |= cmask & ({}u << (r * {}));".format((1 << V) - 1, V), 2)
        e("}")
        full_mask = (1 << (R * V)) - 1
        e("const bool interior = __syncthreads_and(cmask == {}u);".format(full_mask))
        if ndim == 3:
            e("i64 out_off = ((i64)gj0 - (i64)s_base * {NJ}) * {NK} + gk;   // element offset of the thread's first cell in plane 0".format(NJ=self.NJ, NK=self.NK))
        else:
            e("i64 out_off = (i64)gk - (i64)s_base * {NK};".format(NK=self.NK))
        e("asm volatile(\"\" : \"+r\"(cmask), \"+r\"(smask));   // keep them in registers: no re-derivation from blockIdx in the loop")
        if g.unaligned:
            e("asm volatile(\"\" : \"+r\"(stmask));")
        for n in range(len(stored)):
            e("{T}* ob_{n} = o_{n} + out_off;".format(T=T, n=n))
            e("asm volatile(\"\" : \"+l\"(ob_{n}));".format(n=n))
        # lower-dimensional inputs that do not vary along the streamed dimension: loaded once per tile
        self.aux_regs = {}
        for n, (field, off) in enumerate(a.aux_hoisted()):
            self.aux_regs[(field, off)] = self._emit_aux_load(field, off, None, "ax{}".format(n), 1)
        tile_bytes = g.TR * g.TC * self.ct.bytes
        e("const int t_end = c_end + ({});".format(a.t_end_offset()))
        if U > 1:
            # the step count is rounded up to a multiple of the unroll factor by starting earlier:
            # the extra leading steps only produce planes nobody stores or reads
            e("const int t_begin = t_end - ((t_end - (c_begin + ({off})) + {Um1}) / {U}) * {U};".format(
                off=a.t_begin_offset(), Um1=U - 1, U=U))
        else:
            e("const int t_begin = c_begin + ({});".format(a.t_begin_offset()))
        # TMA issue helper as a lambda
        nbox = g.TC // g.box_cols
        nwarps = g.NT // 32
        total_boxes = nbox * len(ext)
        # one elected lane of warp 0 arms the mbarrier; with many boxes per plane (wide 2-D tiles) the
        # copies themselves are issued by the first `issuers` warps, one box each per round
        issuers = 1 if total_boxes <= 2 else min(nwarps, nbox)
        if g.unaligned:
            # every thread of a barrier's group copies its share of the group's part of the plane
            if g.halves:
                e("const u32 upper_u = warp_u >= {} ? 1u : 0u;              // which half of the tile this warp belongs to".format(nwarps // 2))
                e("const u32 seam_lo = warp_u == {} ? 1u : 0u, seam_hi = warp_u == {} ? 1u : 0u;".format(nwarps // 2 - 1, nwarps // 2))
                e("unsigned long long* const wbars = bars + upper_u * {};".format(g.D))
            elif g.pair:
                e("unsigned long long* const wbars = bars + warp_u * {};".format(g.D))
            else:
                e("unsigned long long* const wbars = bars;")
            self._emit_copy_issue(ext)
        elif g.pair:
            # every warp stages its own rows (3-D) / columns (2-D) of the plane and owns the barriers
            box_elems = g.box[0] * g.box[1]
            e("unsigned long long* const wbars = bars + warp_u * {};".format(g.D))
            e("auto issue = [&](int t, int s) {")
            e("sf_mbar_expect_tx(&wbars[s], {});".format(box_elems * self.ct.bytes * len(ext)), 2)
            for n, i in enumerate(ext):
                plane = "t - ({}) - s_base".format(i.lag)
                if ndim == 3:
                    dst = "tile_{f} + s * {sz} + warp_u * {wsz}".format(f=self.fid[i.name], sz=g.TR * g.TC,
                                                                       wsz=g.warp_rows * g.TC)
                    e("sf_tma_load_3d({}, &tm_{}, &wbars[s], tile_k0 - {}, tile_j0 - {} + warp_u * {}, {});".format(
                        dst, n, g.HK0, g.HJ0, g.warp_rows, plane), 2)
                else:
                    dst = "tile_{f} + s * {sz} + warp_u * {wsz}".format(f=self.fid[i.name], sz=g.TR * g.TC,
                                                                       wsz=g.box[0])
                    e("sf_tma_load_2d({}, &tm_{}, &wbars[s], tile_k0 - {} + warp_u * {}, {});".format(
                        dst, n, g.HK0, g.box[0], plane), 2)
            e("};")
            issuers = nwarps
        elif g.halves:
            half_bytes = (g.TR // 2) * g.TC * self.ct.bytes
            e("const u32 upper_u = warp_u >= {} ? 1u : 0u;              // which half of the tile this warp belongs to".format(nwarps // 2))
            e("const u32 seam_lo = warp_u == {} ? 1u : 0u, seam_hi = warp_u == {} ? 1u : 0u;".format(nwarps // 2 - 1, nwarps // 2))
            e("unsigned long long* const wbars = bars + upper_u * {};".format(g.D))
            e("auto issue = [&](int t, int s) {")
            e("sf_mbar_expect_tx(&wbars[s], {});".format(half_bytes * len(ext)), 2)
            for n, i in enumerate(ext):
                plane = "t - ({}) - s_base".format(i.lag)
                dst = "tile_{f} + s * {sz} + upper_u * {hsz}".format(f=self.fid[i.name], sz=g.TR * g.TC,
                                                                     hsz=(g.TR // 2) * g.TC)
                e("sf_tma_load_3d({}, &tm_{}, &wbars[s], tile_k0 - {}, tile_j0 - {} + (int)upper_u * {}, {});".format(
                    dst, n, g.HK0, g.HJ0, g.TR // 2, plane), 2)
            e("};")
            issuers = 0
        else:
            e("unsigned long long* const wbars = bars;")
            e("auto issue = [&](int t, int s) {")
            e("if (warp_u == 0) sf_mbar_expect_tx(&bars[s], {});".format(tile_bytes * len(ext)), 2)
            for n, i in enumerate(ext):
                plane = "t - ({}) - s_base".format(i.lag)
                if issuers == 1:
                    boxes = [str(b * g.box_cols) for b in range(nbox)]
                else:
                    e("for (int b = warp_u; b < {}; b += {}) {{".format(nbox, issuers), 2)
                    boxes = ["b * {}".format(g.box_cols)]
                for bo in boxes:
                    dst = "tile_{f} + s * {sz} + {bo}".format(f=self.fid[i.name], sz=g.TR * g.TC, bo=bo)
                    if ndim == 3:
                        e("sf_tma_load_3d({}, &tm_{}, &bars[s], tile_k0 - {} + {}, tile_j0 - {}, {});".format(
                            dst, n, g.HK0, bo, g.HJ0, plane), 2)
                    else:
                        e("sf_tma_load_2d({}, &tm_{}, &bars[s], tile_k0 - {} + {}, {});".format(
                            dst, n, g.HK0, bo, plane), 2)
                if issuers > 1:
                    e("}", 2)
            e("};")
        if g.unaligned:
            e("const bool issuer = true;                  // (every thread copies its share of a plane)")
        elif g.halves:
            e("const bool issuer = (warp_u % {}) == 0;            // the first warp of each half".format(nwarps // 2))
        else:
            e("const bool issuer = warp_u < {};".format(issuers))
        e("if (issuer) {" if g.unaligned else "if (issuer && sf_elect_one()) {")
        if static_d:
            e("for (int p = 0; p < {}; ++p) if (t_begin + p < t_end) issue(t_begin + p, p);".format(g.P), 2)
        else:
            e("for (int p = 0; p < {P}; ++p) if (t_begin + p < t_end) issue(t_begin + p, (slot + p) % {D});".format(
                P=g.P, D=g.D), 2)
        e("}")
        needs_bc = [i for i in a.fields.values() if self._needs_fixup(i)]
        # ``copy`` boundaries are resolved by the consuming operator: its trips near the border need the code too
        needs_bc += [a.fields[op] for (op, _) in sorted(a.copy_taps) if a.fields[op] not in needs_bc]
        needs_bc += [a.fields[f] for (_, f) in sorted(a.copy_taps) if a.fields[f] not in needs_bc]
        # a trip without boundary code needs the planes of an operator's copy taps inside the domain as well: the
        # operator at plane t - lag reads plane t - lag + d
        back = [i.lag for i in needs_bc] + [a.fields[op].lag - lo for (op, _), (lo, _) in a.copy_reach.items()]
        ahead = [i.lag for i in needs_bc] + [a.fields[op].lag - hi for (op, _), (_, hi) in a.copy_reach.items()]
        def emit_loop(n_ops):
            self.ops_limit = n_ops
            flip = static_d and (U // g.D) % 2 == 1
            if needs_bc and self.fast_path and self.split_loop:
                # a trip whose planes all lie inside the domain, in a CTA whose cells all do, needs no boundary
                # values: it runs a copy of the steps without any of that code.  The two copies are separate
                # loops -- runs of fast trips, single trips with the boundary code in between -- rather than the
                # two arms of a branch inside one loop: the register assignment of the fast loop is then its own
                # (no copies at the join of the arms: 57 MOV per trip of the Jacobi-3D pass)
                lag_max = max(back)
                lag_min = min(ahead)
                cond = "__all_sync(0xffffffffu, interior && (t0 - ({}) >= 0) && (t0 + {} - ({}) < {}))".format(
                    lag_max, U - 1, lag_min, self.NS)
                e("int t0 = t_begin;")
                e("#pragma unroll 1")
                e("while (t0 < t_end) {")
                e("#pragma unroll 1", 2)
                e("while (t0 < t_end && {}) {{".format(cond), 2)
                self.with_bc = False
                self._emit_steps(ext, static_d)
                if flip:
                    e("phase ^= 1u;", 2)
                e("t0 += {};".format(U), 2)
                e("}", 2)
                e("if (t0 < t_end) {", 2)
                self.with_bc = True
                self._emit_steps(ext, static_d)
                if flip:
                    e("phase ^= 1u;", 2)
                e("t0 += {};".format(U), 2)
                e("}", 2)
                e("}")
            else:
                e("#pragma unroll 1")
                e("for (int t0 = t_begin; t0 < t_end; t0 += {}) {{".format(U))
                variants = [True]
                if needs_bc and self.fast_path:
                    lag_max = max(back)
                    lag_min = min(ahead)
                    e("const bool fast = __all_sync(0xffffffffu, interior && (t0 - ({}) >= 0) && (t0 + {} - ({}) < {}));".format(
                        lag_max, U - 1, lag_min, self.NS), 2)
                    variants = [False, True]
                for with_bc in variants:
                    self.with_bc = with_bc
                    if len(variants) == 2:
                        e("if (fast) {" if not with_bc else "} else {", 2)
                    self._emit_steps(ext, static_d)
                if len(variants) == 2:
                    e("}", 2)
                if flip:
                    e("phase ^= 1u;", 2)
                e("}")

        if self.skip_from < len(self.ops):
            # the warps that hold nothing but outer halo rows (see _halo_warps) stream through their own copy
            # of the loop, which runs the leading operators only; barriers are counted, not matched by
            # address, so the two loops meet at every step all the same
            e("if (halo_warp) {")
            emit_loop(self.skip_from)
            e("} else {")
            emit_loop(len(self.ops))
            e("}")
        else:
            emit_loop(len(self.ops))
        if self.peer_push:
            # slab mode: the planes of this segment that a neighbouring GPU reads as halo follow the
            # segment out (all result stores of the CTA are visible to it after the barrier)
            j0 = "tile_j0" if ndim == 3 else "0"
            j1 = "min(tile_j0 + {}, {})".format(g.BJ, self.NJ) if ndim == 3 else "1"
            for n in range(len(stored)):
                e("if (c_begin < pe_lo_{n} || c_end > pb_hi_{n}) {{".format(n=n))
                e("__syncthreads();", 2)
                for (d, lo, hi) in (("pd_lo", "c_begin", "min(c_end, pe_lo_{})".format(n)),
                                    ("pd_hi", "max(c_begin, pb_hi_{})".format(n), "c_end")):
                    e("sf_push_planes<{T}>(o_{n}, {d}_{n}, {lo}, {hi}, s_base, {j0}, {j1}, tile_k0, min(tile_k0 + {BK}, {NK}), {NJ}, {NK});".format(
                        T=T, n=n, d=d, lo=lo, hi=hi, j0=j0, j1=j1, BK=g.BK, NK=self.NK,
                        NJ=self.NJ if ndim == 3 else 1), 2)
                e("}")
        if self.persistent:
            e("__syncthreads();")
            e("if (threadIdx.x == 0) *sf_item = (int)gridDim.x + atomicAdd(&work_tab[0], 1);")
            e("__syncthreads();")
            e("item = *sf_item;")
        e("}   // segment")
        if self.persistent:
            # the last CTA to leave resets the counters for the next launch of this table
            e("if (threadIdx.x == 0) {")
            e("__threadfence();", 2)
            e("if (atomicAdd(&work_tab[1], 1) == (int)gridDim.x - 1) { work_tab[0] = 0; work_tab[1] = 0; __threadfence(); }", 2)
            e("}")
        if self.tmem:
            e("sf_tmem_wait_st();")
            e("sf_tmem_fence_before();")
            e("__syncthreads();")
            e("if (warp_u == 0) { sf_tmem_fence_after(); sf_tmem_dealloc(*sf_tmem); }")
        body = "\n".join(self.lines)
        digest = hashlib.sha1((body + ";".join(params)).encode()).hexdigest()[:12]
        name = "sf_stream_{}".format(digest)
        src = ("extern \"C\" __global__ void __launch_bounds__({}, 1)\n{}({})\n{{\n{}\n}}\n".format(
            g.NT, name, ", ".join(params), body))
        if g.unaligned:
            args = [("buf", i.name) for i in ext]
        else:
            args = [("tmap", {"field": i.name, "box": self._box()}) for i in ext]
        args += [("buf", i.name) for i in stored]
        args += [("buf", name) for name in a.aux]
        args += [("scalar", self.program.fields[s].data_type, s) for s in self.scalars]
        args += [("slab",), ("worktab",) if self.persistent else ("chunk",)]
        if self.peer_push:
            args += [("push", i.name) for i in stored]
        return name, src, args

    def _emit_tmem_alloc(self):
        """Warp 0 allocates the 512 columns; every warp then owns 128 of them in its lane quarter."""
        e = self.emit
        e("if (warp_u == 0) sf_tmem_alloc(sf_tmem);")
        e("sf_tmem_fence_before();")
        e("__syncthreads();")
        e("sf_tmem_fence_after();")
        e("const u32 tm_base = *sf_tmem + ((u32)(32 * (warp_u % 4)) << 16) + (u32)(warp_u / 4) * 128;")

    def _tm_words(self, info, slot):
        """(C lvalues of the cells of a window slot, 32-bit words of them in column order)"""
        g = self.geo
        cells = [self.cellref("w_{}[{}][{}]".format(self.fid[info.name], slot, r), v)
                 for r in range(g.R) for v in range(g.V)]
        if self.ct == dtypes.float32:
            return cells, ["__float_as_uint({})".format(c) for c in cells]
        return cells, [w for c in cells for w in ("(u32)__double2loint({})".format(c), "(u32)__double2hiint({})".format(c))]

    def _tm_chunks(self, n):
        pos = 0
        for size in (16, 8, 4, 2, 1):
            while n - pos >= size:
                yield pos, size
                pos += size

    def _tm_column(self, name, parity):
        return "tm_base + {}".format((2 * list(self.ana.tmem_ages).index(name) + parity) * self.geo.tmem_cols)

    def _tm_store(self, info, u):
        """Parks the plane that is one step younger than the field's TMEM slot (its last use is behind it)."""
        age = self.ana.tmem_ages[info.name]
        cells, words = self._tm_words(info, self.wslot(info, age - 1, u))
        col = self._tm_column(info.name, (u - age + 1) % 2)
        for pos, n in self._tm_chunks(len(words)):
            self.emit("sf_tmem_st{}({} + {}, {});".format(n, col, pos, ", ".join(words[pos:pos + n])), 2)

    def _tm_load(self, info, u):
        """Fetches the field's TMEM slot back into its window registers (valid after _tm_wait)."""
        e = self.emit
        age = self.ana.tmem_ages[info.name]
        cells, words = self._tm_words(info, self.wslot(info, age, u))
        col = self._tm_column(info.name, (u - age) % 2)
        e("{", 3)
        e("u32 tl[{}];".format(len(words)), 4)
        for pos, n in self._tm_chunks(len(words)):
            e("sf_tmem_ld{}({} + {}, {});".format(n, col, pos, ", ".join("tl[{}]".format(pos + i) for i in range(n))), 4)
        for i, c in enumerate(cells):
            if self.ct == dtypes.float32:
                e("{} = __uint_as_float(tl[{}]);".format(c, i), 4)
            else:
                e("{} = __hiloint2double((int)tl[{}], (int)tl[{}]);".format(c, 2 * i + 1, 2 * i), 4)
        e("}", 3)

    def _tm_wait(self, info, u):
        """tcgen05.wait::ld, then an empty asm that takes the loaded registers through it, so that the
        compiler does not move their first use above the wait"""
        age = self.ana.tmem_ages[info.name]
        cells, _ = self._tm_words(info, self.wslot(info, age, u))
        self.emit("sf_tmem_wait_ld();", 3)
        c = "f" if self.ct == dtypes.float32 else "d"
        for pos in range(0, len(cells), 16):
            self.emit("asm volatile(\"\" : {});".format(", ".join('"+{}"({})'.format(c, x) for x in cells[pos:pos + 16])), 3)

    def _tm_store_points(self, ops):
        """{position: [fields]} where the step parks each TMEM field: after the last of ``ops`` that reads the
        plane one step younger than its slot (k), after the streamed inputs (-1) or at the start of the step (-2)"""
        a = self.ana
        out = collections.defaultdict(list)
        names = [op.name for op in ops]
        for name, age in (a.tmem_ages.items() if self.tmem else []):
            src = a.fields[name]
            readers = [k for k, op in enumerate(ops) for (f, d, dj, dk) in a.taps[op.name]
                       if f == name and a.fields[op.name].lag - d - src.lag == age - 1]
            if readers:
                out[max(readers)].append(src)
            elif age > 1:
                out[-2].append(src)
            elif src.kind == "ext":
                out[-1].append(src)
            elif name in names:
                out[names.index(name)].append(src)
        return out

    def _needs_fixup(self, info):
        """Cells outside the domain must read as the boundary value.  Input planes arrive through TMA,
        which zero-fills everything outside the tensor, so a zero boundary value needs no code -- except with
        unaligned rows: the cell copies only zero-fill past the ends of the whole array, and the cells left and
        right of a row and in the rows beyond the domain's edges hold neighbouring rows' data."""
        if not info.consumed or info.bc is None:
            return False
        return not (info.kind == "ext" and float(info.bc) == 0.0 and not self.geo.unaligned)

    def _copy_threads(self):
        """Unaligned rows: (threads that copy for one mbarrier, C expression of a thread's rank among them)."""
        g = self.geo
        if g.pair:
            return 32, "(int)(threadIdx.x & 31)"
        if g.halves:
            return g.NT // 2, "(int)(threadIdx.x % {})".format(g.NT // 2)
        return g.NT, "(int)threadIdx.x"

    def _emit_copy_issue(self, ext):
        """Unaligned rows: ``issue(t, s)`` copies the cells of every streamed input's plane that the calling thread's
        mbarrier group stages (the whole tile; a warp's rows or columns with ``pair``; a half's rows with
        ``halves``) into ring slot s, one ``cp.async`` per cell, the threads of the group taking turns.  Cells
        outside the array are zero-filled; a thread arrives on the slot's mbarrier once its copies have landed.
        Row starts are anywhere in memory, so no copy wider than a cell is aligned in general.  (One rank-1 TMA
        box per tile row, started at such an address, stopped the first kernel that used it with an illegal
        instruction on a B200: DESIGN 3.2.)"""
        g, a, e = self.geo, self.ana, self.emit
        nthr, tid = self._copy_threads()
        if g.pair and a.ndim == 3:
            row0, nrows, col0, ncols = "warp_u * {}".format(g.warp_rows), g.warp_rows, "0", g.TC
        elif g.pair:
            row0, nrows, col0, ncols = "0", 1, "warp_u * {}".format(g.box[0]), g.box[0]
        elif g.halves:
            row0, nrows, col0, ncols = "(int)upper_u * {}".format(g.TR // 2), g.TR // 2, "0", g.TC
        else:
            row0, nrows, col0, ncols = "0", (g.TR if a.ndim == 3 else 1), "0", g.TC
        plane = self.NJ * self.NK if a.ndim == 3 else self.NK
        e("auto issue = [&](int t, int s) {")
        for n, i in enumerate(ext):
            e("{", 2)
            if a.ndim == 3:
                e("const i64 pb = (i64)(t - ({lag}) - s_base) * {pl} + (i64)(tile_j0 - {HJ0} + {row0}) * {NK} + tile_k0 - {HK0} + {col0};".format(
                    lag=i.lag, pl=plane, HJ0=g.HJ0, row0=row0, NK=self.NK, HK0=g.HK0, col0=col0), 3)
            else:
                e("const i64 pb = (i64)(t - ({lag}) - s_base) * {pl} + tile_k0 - {HK0} + {col0};".format(
                    lag=i.lag, pl=plane, HK0=g.HK0, col0=col0), 3)
            e("#pragma unroll 1", 3)
            e("for (int q = {tid}; q < {n}; q += {nthr}) {{".format(tid=tid, n=nrows * ncols, nthr=nthr), 3)
            e("const int r = q / {c}, c = q - r * {c};".format(c=ncols), 4)
            e("sf_cp_async(tile_{f} + s * {sz} + ({row0} + r) * {TC} + {col0} + c, in_{n}, pb + (i64)r * {NK} + c, {tot}ll);".format(
                f=self.fid[i.name], sz=g.TR * g.TC, row0=row0, TC=g.TC, col0=col0, n=n, NK=self.NK,
                tot=self.NS * plane), 4)
            e("}", 3)
            e("}", 2)
        e("sf_cp_async_arrive(&wbars[s]);", 2)
        e("};")

    def _emit_steps(self, ext, static_d):
        g, a, e, U = self.geo, self.ana, self.emit, self.U
        for u in range(U):
            e("{{  // ---- unrolled step {}".format(u), 2)
            e("const int t = t0 + {};".format(u), 2)
            if static_d:
                self.slot_expr = str(u % g.D)
                nxt = str((u + g.P) % g.D)
                ph = "phase" if (u // g.D) % 2 == 0 else "(phase ^ 1u)"
            else:
                self.slot_expr = "slot"
                nxt = "(slot + {P}) % {D}".format(P=g.P, D=g.D)
                ph = "phase"
            self._waited = set()
            self._tm_loaded, self._tm_waited = set(), set()
            if self.tmem:
                # the stores of the previous step land before this step fetches what they parked
                e("sf_tmem_wait_st();", 2)
            if self.flags:
                # every warp has read its rows of the plane in the TMA slot about to be refilled once it has
                # published them: the arrivals of the previous step on the streamed inputs' barriers
                for i in ext:
                    self._flag_wait(i, 1, u)
            if g.unaligned:
                e("if (issuer && t + {P} < t_end) issue(t + {P}, {nxt});".format(P=g.P, nxt=nxt), 2)
            else:
                e("if (issuer && t + {P} < t_end) {{ if (sf_elect_one()) issue(t + {P}, {nxt}); }}".format(P=g.P, nxt=nxt), 2)
            last_comm = self._emit_ops(u, ext, ph, self.ops_limit)
            if g.pair:
                e("sf_sync_neighbours<{}>(warp_u);".format(g.NW), 2)
            elif g.halves:
                # (barrier ids alternate with the step so that a half one step ahead cannot arrive twice on one id)
                ids = (3, 4) if u % 2 == 0 else (5, 6)
                e("sf_seam_handshake<{}, {}>(seam_lo, seam_hi);".format(*ids), 2)
                e("sf_bar_half(upper_u, {}u);".format(g.NT // 2), 2)
            elif self.flags:
                pass
            elif self.split_barrier:
                self.lines.insert(last_comm, "  " * 2 + "__syncwarp(); if (sf_elect_one()) sf_mbar_arrive(sbar);")
                # (segments are whole trips of U steps: with an even U the phase of a step is static)
                if U % 2:
                    e("sf_mbar_wait(sbar, sphase); sphase ^= 1u;", 2)
                else:
                    e("sf_mbar_wait(sbar, {}u);".format(u % 2), 2)
            else:
                e("__syncthreads();", 2)
            if not static_d:
                e("if (++slot == {}) {{ slot = 0; phase ^= 1; }}".format(g.D), 2)
            for i in a.fields.values():
                if i.row_ring and i.name not in g.direct and not self.static(i.row_ring):
                    e("if (++xr_{f} == {n}) xr_{f} = 0;".format(f=self.fid[i.name], n=i.row_ring), 2)
                if i.col_ring and not self.static(i.col_ring):
                    e("if (++xc_{f} == {n}) xc_{f} = 0;".format(f=self.fid[i.name], n=i.col_ring), 2)
            e("}", 2)

    def _emit_ops(self, u, ext, ph, n_ops):
        """One streamed step of a thread: the new plane of every input, then the first ``n_ops`` operators.
        Returns the position (in ``self.lines``) after the last shared-memory read / write of the step."""
        g, a, e = self.geo, self.ana, self.emit
        ops = self.ops[:n_ops]
        gathered = {}
        tm_store = self._tm_store_points(ops)
        for info in tm_store.get(-2, []):
            self._tm_store(info, u)
        if ops and self.pipeline and self._can_gather_early(ops[0]):
            # neighbour data of the first operator is a step old: fetch it while the TMA lands
            gathered[0] = self._gather_op(ops[0], u, 0)
        e("sf_mbar_wait(&wbars[{}], {});".format(self.slot_expr, ph), 2)
        for i in ext:
            self._produce_ext(i, u)
        for info in tm_store.get(-1, []):
            self._tm_store(info, u)
        last_comm = len(self.lines)
        for k, op in enumerate(ops):
            if k not in gathered:
                gathered[k] = self._gather_op(op, u, k)
                last_comm = len(self.lines)
            if self.pipeline and k + 1 < len(ops) and self._can_gather_early(ops[k + 1]):
                # software pipelining: the shuffles / ring loads of the next operator are issued
                # before this operator's arithmetic, which hides their latency
                gathered[k + 1] = self._gather_op(ops[k + 1], u, k + 1)
                last_comm = len(self.lines)
            self._produce_op(op, u, gathered.pop(k))
            for src in tm_store.get(k, []):
                self._tm_store(src, u)
            info = a.fields[op.name]
            if info.consumed and (info.row_ring or info.col_ring):
                last_comm = len(self.lines)
        return last_comm

    def _halo_warps(self):
        """3-D tiles: (rotate, warps, first skipped operator).  The outermost halo rows of a tile only feed the
        first operators of the group -- with a halo of 4 rows and 3 rows per thread, rows 0-2 and TR-3..TR-1 are
        read by the first two of four chained operators and by nothing after.  When the row groups are dealt
        to the warps *rotated by one* (two groups per warp at 16 threads per row: warp 0 then holds the last and
        the first group, i.e. only such rows), that warp can leave a step early: it skips the remaining
        operators, whose results on its rows nobody stores or reads for a stored cell (1/24 of the arithmetic
        and exchange traffic of the Jacobi-3D pass).  With a warp per row group the first and the last warp
        qualify without rotation."""
        g, a = self.geo, self.ana
        none = (False, [], len(self.ops))
        if a.ndim != 3 or g.WC != 1 or g.pair or os.environ.get("SFB200_HALO_SKIP", HALO_SKIP_DEFAULT) == "0":
            return none
        if self.flags or self.split_barrier or g.halves or g.NT % 32 or 32 % g.KS:
            return none
        gpw = 32 // g.KS
        best = none
        for rot in ((False, True) if gpw > 1 else (False,)):
            per_warp = {}
            for hw in range(g.NT // 32):
                groups = [((hw * gpw + h) + (g.WR - 1 if rot else 0)) % g.WR for h in range(gpw)]
                first_unneeded = len(self.ops)
                for k in range(len(self.ops) - 1, -1, -1):
                    info = a.fields[self.ops[k].name]
                    lo, hi = g.HJ0 - info.need[0], g.TR - g.HJ1 + info.need[1]
                    if any(lo <= wr * g.R + r < hi for wr in groups for r in range(g.R)):
                        break
                    first_unneeded = k
                per_warp[hw] = first_unneeded
            cut = min(per_warp.values())
            warps = [hw for hw, k in per_warp.items() if k == cut]
            if cut < len(self.ops) and (best[2] == len(self.ops) or
                                         (len(self.ops) - cut) * len(warps) > (len(self.ops) - best[2]) * len(best[1])):
                best = (rot, warps, cut)
        return best

    def _box(self):
        return list(self.geo.box)

    # ------------------------------------------------------------------ producing a field
    def _open_plane(self, info: _FieldInfo, u: int):
        """Declares ``nv``, the R x V cells of the plane being produced: the window slot that becomes
        age 0 (rotating the window by moves only when its period does not divide the unroll factor)."""
        g, e = self.geo, self.emit
        f = self.fid[info.name]
        if not info.consumed:
            e("{ET} nv[{R}][{VH}];".format(ET=self.ET, R=g.R, VH=self.VH), 3)
            return
        if self.wperiod(info) == 0:
            for wdx in range(info.window - 1, 0, -1):
                e("#pragma unroll", 3)
                e("for (int r = 0; r < {}; ++r)".format(g.R), 3)
                e("#pragma unroll", 4)
                e("for (int v = 0; v < {VH}; ++v) w_{f}[{a}][r][v] = w_{f}[{b}][r][v];".format(
                    VH=self.VH, f=f, a=wdx, b=wdx - 1), 4)
        e("{ET} (&nv)[{R}][{VH}] = w_{f}[{s}];".format(ET=self.ET, R=g.R, VH=self.VH, f=f,
                                                      s=self.wslot(info, 0, u)), 3)

    def _finish_field(self, info: _FieldInfo, plane_expr: str, u: int):
        """``nv`` holds the new plane: apply the boundary value, publish the edge rows/columns."""
        g, e = self.geo, self.emit
        f = self.fid[info.name]
        V, R = g.V, g.R
        if not info.consumed:
            return
        if self.with_bc and self._needs_fixup(info):
            e("{")
            e("const bool pin = (unsigned)({}) < {}u;".format(plane_expr, self.NS), 3)
            full = (1 << (R * V)) - 1
            bc = self.lit(info.bc)

            def fix(r, v, ind):
                e("{c} = {bc};".format(c=self.cellref("nv[{}]".format(r), v), bc=bc), ind)

            # one in-domain bit per owned cell.  "thread": only warps that own cells outside the domain
            # (or a plane outside it) enter, and a thread whose cells are all outside overwrites them
            # without testing each one; "cta": every warp of a tile that has any such cell tests every cell
            if self.bc_mode == "thread":
                e("if (!(pin && cmask == {}u)) {{".format(full), 3)
                e("const u32 m = pin ? cmask : 0u;", 4)
                e("if (m == 0u) {", 4)
                for r in range(R):
                    for v in range(V):
                        fix(r, v, 5)
                e("} else {", 4)
                for r in range(R):
                    for v in range(V):
                        e("if (!((m >> {b}) & 1u)) {c} = {bc};".format(
                            b=r * V + v, c=self.cellref("nv[{}]".format(r), v), bc=bc), 5)
                e("}", 4)
                e("}", 3)
            else:
                e("if (!(pin && interior)) {", 3)
                e("const u32 m = pin ? cmask : 0u;", 4)
                for r in range(R):
                    for v in range(V):
                        e("if (!((m >> {b}) & 1u)) {c} = {bc};".format(
                            b=r * V + v, c=self.cellref("nv[{}]".format(r), v), bc=bc), 4)
                e("}", 3)
            e("}")
        if info.row_ring and info.name not in g.direct:
            n = info.row_reach
            # layout [ring][WR][2][n][TC]
            slot = self.ring_slot("xr_" + f, info.row_ring, 0, u)
            base = "xrow_{f} + (({slot} * {WR} + wr) * 2) * {sz}".format(f=f, slot=slot, WR=g.WR, sz=n * g.TC)
            for q in range(n):
                e(self.stv("{base} + {o} + c0".format(base=base, o=q * g.TC), "nv[{}]".format(q)), 2)
                e(self.stv("{base} + {o} + c0".format(base=base, o=(n + q) * g.TC), "nv[{}]".format(R - n + q)), 2)
        if info.col_ring:
            # layout [ring][WR][WC][2][R][n]: the n = col_reach edge cells of every owned row, left
            # edge (side 0, written by lane 0) and right edge (side 1, written by lane 31)
            n = info.col_reach
            slot = self.ring_slot("xc_" + f, info.col_ring, 0, u)
            base = "xcol_{f} + ((({slot} * {WR} + wr) * {WC} + wc) * 2) * {sz}".format(
                f=f, slot=slot, WR=g.WR, WC=g.WC, sz=R * n)
            for r in range(R):
                for q in range(n):
                    e("sf_sts_if(lane == 0 && wc > 0, {base} + {o}, {c});".format(
                        base=base, o=r * n + q, c=self.cellref("nv[{}]".format(r), q)), 2)
            for r in range(R):
                for q in range(n):
                    e("sf_sts_if(lane == 31 && wc < {last}, {{base}} + {{o}}, {{c}});".format(last=g.WC - 1).format(
                        base=base, o=(R + r) * n + q, c=self.cellref("nv[{}]".format(r), V - n + q)), 2)
        if self._published(info):
            self._flag_arrive(info)

    # ------------------------------------------------------------------ lower-dimensional inputs
    def _aux_bc(self, field):
        """Value an out-of-domain tap of ``field`` reads (``cpu.py:73-102``), or None if no tap can."""
        return self.ana.aux_bc.get(field)

    def _emit_aux_load(self, field, off, plane, name, indent, bc=None):
        """Declares ``name`` and loads into it what one tap of a lower-dimensional input reads for the
        thread's cells: ``name[rows][V/G]`` (packed like every other value) when the field varies along
        k, ``name[rows]`` otherwise; rows = R if it varies along the row dimension, else 1.  Indices are
        clamped into the (slab-local) array, positions outside the domain read the boundary value.
        Returns (name, has_row, has_col)."""
        a, g, e, T = self.ana, self.geo, self.emit, self.T
        f = a.aux[field]
        ds, dr, dc = a.aux_split(off)
        it_s, it_r = self.program.iterators[0], ("j" if a.ndim == 3 else None)
        ext = self.program.extents
        strides, stride = {}, 1
        for d in reversed(f.dims):
            strides[d] = stride
            stride *= ext[d]
        has_r, has_c = dr is not None, dc is not None
        RR = g.R if has_r else 1
        bcv = bc if bc is not None else self._aux_bc(field)
        px = self.aux_name[field]
        if has_c:
            e("{ET} {n}[{RR}][{VH}];".format(ET=self.ET, n=name, RR=RR, VH=self.VH), indent)
        else:
            e("{T} {n}[{RR}];".format(T=T, n=name, RR=RR), indent)
        fwd = max([i.fwd for i in a.ext_fields] + [r[1] for r in a.aux_reach.values()])
        for r in range(RR):
            for v in range(g.V if has_c else 1):
                terms, conds = [], []
                if ds is not None:
                    pos = "({} + ({}))".format(plane, ds)
                    hi = "min({}, s_end + {}) - 1".format(self.NS, fwd)
                    terms.append("(i64)(min(max({p}, s_base), {hi}) - s_base) * {st}".format(p=pos, hi=hi, st=strides[it_s]))
                    if ds:
                        conds.append("(unsigned){} < {}u".format(pos, self.NS))
                if has_r:
                    pos = "(gj0 + ({}))".format(r + dr)
                    terms.append("(i64)min(max({p}, 0), {n}) * {st}".format(p=pos, n=self.NJ - 1, st=strides[it_r]))
                    if dr:
                        conds.append("(unsigned){} < {}u".format(pos, self.NJ))
                if has_c:
                    pos = "(gk + ({}))".format(v + dc)
                    terms.append("(i64)min(max({p}, 0), {n}) * {st}".format(p=pos, n=self.NK - 1, st=strides["k"]))
                    if dc:
                        conds.append("(unsigned){} < {}u".format(pos, self.NK))
                load = "__ldg({} + ({}))".format(px, " + ".join(terms))
                if conds:
                    load = "(({}) ? {} : {})".format(" && ".join(conds), load, self.lit(bcv if bcv is not None else 0.0))
                dst = "{}[{}]".format(name, r)
                if has_c:
                    dst = self.cellref(dst, v)
                e("{} = {};".format(dst, load), indent)
        return name, has_r, has_c

    def _aux_key(self, t: ex.Tap):
        dims = self.ana.aux[t.field].dims
        return (t.field, tuple(o if it in dims else None for it, o in zip(ex.ITERATORS, t.offset)))

    def _aux_value(self, regs, r, v):
        """C expression of cell v of row r of a loaded lower-dimensional tap (scalar form)."""
        name, has_r, has_c = regs
        row = "{}[{}]".format(name, r if has_r else 0)
        return self.cellref(row, v) if has_c else row

    def _produce_ext(self, info: _FieldInfo, u: int):
        g, e = self.geo, self.emit
        f = self.fid[info.name]
        e("{  // input field " + f, 2)
        self._open_plane(info, u)
        for r in range(g.R):
            row = "(r0 + {})".format(r) if self.ana.ndim == 3 else "0"
            e(self.ldv("nv[{}]".format(r), "tile_{f} + {slot} * {sz} + {row} * {TC} + c0".format(
                f=f, slot=self.slot_expr, sz=g.TR * g.TC, row=row, TC=g.TC)), 3)
        self._finish_field(info, "t - ({})".format(info.lag), u)
        e("}", 2)

    def _can_gather_early(self, op: StencilOp):
        """True when the operator's neighbour data (shuffled cells, ring rows) can be fetched before
        its sources are produced in the current step: exchange taps are at least one step old by
        construction, so only move-rotated windows (whose slots shift at production) forbid it."""
        a = self.ana
        info = a.fields[op.name]
        for (field, d, dj, dk) in a.taps[op.name]:
            src = a.fields[field]
            if dj == 0 and dk == 0:
                continue
            if info.lag - d - src.lag < 1:
                return False        # shuffles of the plane produced in this very step
            if self.wperiod(src) == 0:
                return False
        return True

    def _gather_op(self, op: StencilOp, u: int, k: int):
        """Emits the loads of everything operator ``op`` reads from other threads (warp shuffles for
        k-neighbours, exchange-ring rows for j-neighbours) and returns the naming tables."""
        g, a, e = self.geo, self.ana, self.emit
        info = a.fields[op.name]
        V, R, T = g.V, g.R, self.T
        taps = a.taps[op.name]
        # row vectors needed: (field, age, row) ; shifts needed per row vector
        rows = collections.OrderedDict()
        for (field, d, dj, dk) in taps:
            src = a.fields[field]
            age = info.lag - d - src.lag
            for r in range(R):
                key = (field, age, r + dj)
                ent = rows.setdefault(key, [0, 0])
                if dk < 0:
                    ent[0] = max(ent[0], -dk)
                if dk > 0:
                    ent[1] = max(ent[1], dk)
        names = {}
        for (field, age, rr), (nl, nr) in rows.items():
            src = a.fields[field]
            f = self.fid[field]
            tag = "o{}_{}_{}_{}".format(k, f, age, _fmt_off(rr))
            if self.tmem and a.tmem_ages.get(field) == age and field not in self._tm_loaded:
                self._tm_loaded.add(field)
                self._tm_load(src, u)
            if not (0 <= rr < R) or (src.col_ring and (nl or nr)):
                self._flag_wait(src, age, u, 3)
            if 0 <= rr < R:
                vec = "w_{}[{}][{}]".format(f, self.wslot(src, age, u), rr)
                names[(field, age, rr)] = (vec, tag)
                if nl or nr:
                    self._emit_shifts(src, vec, tag, rr, age, nl, nr, u)
            else:
                # a row owned by the neighbouring warp: read it (and its shifted columns) from the ring
                n = src.row_reach
                if field in g.direct:
                    # ... or, for a streamed input, from the plane itself in the TMA ring (rows beyond
                    # the tile belong to halo cells nobody uses: clamp them into the tile)
                    slot = (u - age) % g.D
                    row = "max(r0 - {}, 0)".format(-rr) if rr < 0 else "min(r0 + {}, {})".format(rr, g.TR - 1)
                    base = "tile_{f} + {slot} * {sz} + {row} * {TC}".format(f=f, slot=slot, sz=g.TR * g.TC,
                                                                         row=row, TC=g.TC)
                    e("const {T}* const p_{tag} = {base};".format(T=T, tag=tag, base=base), 3)
                    e("{ET} x_{tag}[{VH}];".format(ET=self.ET, tag=tag, VH=self.VH), 3)
                    e(self.ldv("x_" + tag, "p_{} + c0".format(tag)), 3)
                    names[(field, age, rr)] = ("x_" + tag, tag)
                    if nl:
                        e("{T} l_{tag}[{n}];".format(T=T, tag=tag, n=nl), 3)
                        for q in range(nl):
                            e("l_{tag}[{q}] = p_{tag}[max(c0 - {nl} + {q}, 0)];".format(tag=tag, q=q, nl=nl), 3)
                    if nr:
                        e("{T} g_{tag}[{n}];".format(T=T, tag=tag, n=nr), 3)
                        for q in range(nr):
                            e("g_{tag}[{q}] = p_{tag}[min(c0 + {V} + {q}, {last})];".format(
                                tag=tag, q=q, V=V, last=g.TC - 1), 3)
                    continue
                slot = self.ring_slot("xr_" + f, src.row_ring, age, u)
                if rr < 0:
                    nbr = "max(wr - 1, 0)"
                    side_row = n + (n + rr)          # bottom rows of the warp above
                else:
                    nbr = "min(wr + 1, {})".format(g.WR - 1)
                    side_row = rr - R                # top rows of the warp below
                base = "xrow_{f} + (({slot} * {WR} + {nbr}) * 2) * {sz} + {o}".format(
                    f=f, slot=slot, WR=g.WR, nbr=nbr, sz=n * g.TC, o=side_row * g.TC)
                e("const {T}* const p_{tag} = {base};".format(T=T, tag=tag, base=base), 3)
                e("{ET} x_{tag}[{VH}];".format(ET=self.ET, tag=tag, VH=self.VH), 3)
                e(self.ldv("x_" + tag, "p_{} + c0".format(tag)), 3)
                names[(field, age, rr)] = ("x_" + tag, tag)
                if nl:
                    e("{T} l_{tag}[{n}];".format(T=T, tag=tag, n=nl), 3)
                    for q in range(nl):
                        e("l_{tag}[{q}] = p_{tag}[max(c0 - {nl} + {q}, 0)];".format(tag=tag, q=q, nl=nl), 3)
                if nr:
                    e("{T} g_{tag}[{n}];".format(T=T, tag=tag, n=nr), 3)
                    for q in range(nr):
                        e("g_{tag}[{q}] = p_{tag}[min(c0 + {V} + {q}, {last})];".format(
                            tag=tag, q=q, V=V, last=g.TC - 1), 3)
        return rows, names

    def _produce_op(self, op: StencilOp, u: int, gathered):
        g, a, e = self.geo, self.ana, self.emit
        info = a.fields[op.name]
        V, R, T = g.V, g.R, self.T
        plane = "t - ({})".format(info.lag)
        rows, names = gathered
        e("{  // operator producing " + self.fid[op.name], 2)

        def tap_key(t: ex.Tap, r: int):
            if a.ndim == 3:
                d, dj, dk = t.offset
            else:
                d, dj, dk = t.offset[1], 0, t.offset[2]
            src = a.fields[t.field]
            age = info.lag - d - src.lag
            return (t.field, age, r + dj), dk

        def raw_cell(t: ex.Tap, r: int, c: int) -> str:
            key, _ = tap_key(t, r)
            vec, tag = names[key]
            nl, nr = rows[key]
            if 0 <= c < V:
                return self.cellref(vec, c)
            if c < 0:
                return "l_{}[{}]".format(tag, nl + c)
            return "g_{}[{}]".format(tag, c - V)

        copy_fields = {f for (o, f) in a.copy_taps if o == op.name} if self.with_bc else set()

        def tap_cell(t: ex.Tap, r: int, c: int) -> str:
            """C expression of the cell at column c (relative to the thread's first cell); a ``copy`` tap
            that leaves the domain reads the field's centre tap at the cell being computed instead"""
            text = raw_cell(t, r, c)
            if t.field not in copy_fields:
                return text
            if a.ndim == 3:
                d, dj, dk = t.offset
            else:
                d, dj, dk = t.offset[1], 0, t.offset[2]
            if (d, dj, dk) == (0, 0, 0):
                return text
            v = c - dk                                   # the cell of this thread being computed
            conds = []
            if d:
                conds.append("(unsigned)(({}) + ({})) < {}u".format(plane, d, self.NS))
            if dj:
                conds.append("(unsigned)(gj0 + ({})) < {}u".format(r + dj, self.NJ))
            if dk:
                conds.append("(unsigned)(gk + ({})) < {}u".format(c, self.NK))
            centre = raw_cell(ex.Tap(t.field, (0, 0, 0)), r, v)
            return "(({}) ? {} : {})".format(" && ".join(conds), text, centre)

        # lower-dimensional inputs: taps that vary along the streamed dimension are loaded per plane
        self.aux_cur = {}
        for n, (field, off) in enumerate(a.aux_taps.get(op.name, [])):
            if (field, off) in self.aux_cur:
                continue
            if (field, off) in self.aux_regs:
                self.aux_cur[(field, off)] = self.aux_regs[(field, off)]
            else:
                self.aux_cur[(field, off)] = self._emit_aux_load(field, off, "(" + plane + ")", "ay{}".format(n), 3)
        self._open_plane(info, u)
        for (field, age, rr) in rows:
            if self.tmem and a.tmem_ages.get(field) == age and field not in self._tm_waited:
                self._tm_waited.add(field)
                self._tm_wait(a.fields[field], u)
        if self.G == 1:
            self._emit_scalar_cells(op, tap_key, tap_cell)
        else:
            self._emit_packed_cells(op, names, tap_key, tap_cell)
        if info.stored:
            idx = [i.name for i in a.fields.values() if i.stored].index(op.name)
            e("{T}* op = ob_{n} + (i64)({p}) * {stride};".format(
                T=T, n=idx, p=plane, stride=(self.NJ * self.NK if a.ndim == 3 else self.NK)), 3)
            e("asm volatile(\"\" : \"+l\"(op));              // one address computation for all rows", 3)
            e("const bool inchunk = ({p}) >= c_begin && ({p}) < c_end;".format(p=plane), 3)
            if g.unaligned:
                for r in range(R):
                    for v in range(V):
                        e("sf_stg1_if(inchunk && ((stmask >> {b}) & 1u), op + {o}, {c});".format(
                            b=r * V + v, o=r * self.NK + v, c=self.cellref("nv[{}]".format(r), v)), 3)
            else:
                for r in range(R):
                    e("sf_stg_if(inchunk && ({sm} & {m}u), op + {o}, nv[{r}]);".format(
                        sm="smask", m=1 << r, o=r * self.NK, r=r), 3)
        self._finish_field(info, plane, u)
        e("}", 2)

    # ------------------------------------------------------------------ expressions, one cell at a time
    def _emit_scalar_cells(self, op, tap_key, tap_cell):
        g, e, T = self.geo, self.emit, self.T
        math_fn = _MATH_F32 if self.ct == dtypes.float32 else _MATH_F64
        local_ids = {}
        for r in range(g.R):
            for v in range(g.V):
                local = {}
                assigned = collections.Counter()
                for s in op.statements:
                    rhs = ex.emit_c(
                        s.value,
                        tap=lambda t, r=r, v=v: (self._aux_value(self.aux_cur[self._aux_key(t)], r, v)
                                                 if t.field in self.ana.aux else tap_cell(t, r, v + tap_key(t, r)[1])),
                        var=lambda n, local=local: self._var(n, local, op),
                        literal=self.lit,
                        call=lambda fn, args: "{}({})".format(math_fn[fn], ", ".join(args)))
                    if s.target not in local_ids:
                        local_ids[s.target] = len(local_ids)
                    lname = "q{}_{}_{}".format(local_ids[s.target], r, v)
                    ty = "const bool" if isinstance(s.value, (ex.Cmp, ex.Logic)) else "const " + T
                    # a fresh name per assignment: q..., q...b, q...b2, ...
                    n = assigned[s.target]
                    if n:
                        lname += "b" if n == 1 else "b{}".format(n)
                    assigned[s.target] += 1
                    e("{} {} = {};".format(ty, lname, rhs), 3)
                    local[s.target] = lname
                target = op.name if op.name in local else op.statements[-1].target
                e("{} = {};".format(self.cellref("nv[{}]".format(r), v), local[target]), 3)

    # ------------------------------------------------------------------ expressions, two cells at a time
    def _emit_packed_cells(self, op, names, tap_key, tap_cell):
        """float32: every value is a pair of neighbouring cells (2h, 2h+1) of one row.

        Value kinds: ("p", float2 lvalue) | ("s", lo, hi) scalar float expressions that do not form an
        aligned register pair | ("c", uniform scalar expression) | ("b", lo, hi) boolean lanes |
        ("cb", uniform boolean)."""
        g, e, V = self.geo, self.emit, self.geo.V
        math_fn = _MATH_F32

        for r in range(g.R):
            for h in range(V // 2):
                local = {}

                def lanes(v):
                    if v[0] == "p":
                        return v[1] + ".x", v[1] + ".y"
                    if v[0] in ("c", "cb"):
                        return v[1], v[1]
                    return v[1], v[2]

                def as_pair(v):
                    if v[0] == "p":
                        return v[1]
                    assert v[0] == "c"
                    return "make_float2({0}, {0})".format(v[1])

                def new_pair(lo, hi):
                    n = self.tmp()
                    e("float2 {n}; {n}.x = {lo}; {n}.y = {hi};".format(n=n, lo=lo, hi=hi), 3)
                    return ("p", n)

                def packed(fn, *vals):
                    n = self.tmp()
                    e("const float2 {n} = {fn}({args});".format(n=n, fn=fn, args=", ".join(as_pair(v) for v in vals)), 3)
                    return ("p", n)

                def packable(*vals):
                    return all(v[0] in ("p", "c") for v in vals) and any(v[0] == "p" for v in vals)

                def negc(v):
                    return ("c", "(-{})".format(v[1]))

                def val(x):
                    if isinstance(x, ex.Const):
                        if isinstance(x.value, bool):
                            return ("cb", "true" if x.value else "false")
                        return ("c", self.lit(x.value))
                    if isinstance(x, ex.Var):
                        if x.name in local:
                            return local[x.name]
                        return ("c", self._var(x.name, {}, op))
                    if isinstance(x, ex.Tap) and x.field in self.ana.aux:
                        name, has_r, has_c = self.aux_cur[self._aux_key(x)]
                        row = "{}[{}]".format(name, r if has_r else 0)
                        return ("p", "{}[{}]".format(row, h)) if has_c else ("c", row)
                    if isinstance(x, ex.Tap):
                        key, dk = tap_key(x, r)
                        vec, tag = names[key]
                        c = 2 * h + dk
                        plain = not (self.with_bc and (op.name, x.field) in self.ana.copy_taps
                                     and any(x.offset))
                        if plain and dk % 2 == 0 and 0 <= c and c + 1 < V:
                            return ("p", "{}[{}]".format(vec, c // 2))
                        return ("s", tap_cell(x, r, c), tap_cell(x, r, c + 1))
                    if isinstance(x, ex.Bin):
                        if x.op in "+-":
                            fused = fma(x)
                            if fused is not None:
                                return fused
                        va, vb = val(x.a), val(x.b)
                        if va[0] == "c" and vb[0] == "c":
                            return ("c", "({} {} {})".format(va[1], x.op, vb[1]))
                        if x.op in "+-*" and packable(va, vb):
                            return packed({"+": "sf_add2", "-": "sf_sub2", "*": "sf_mul2"}[x.op], va, vb)
                        (alo, ahi), (blo, bhi) = lanes(va), lanes(vb)
                        return new_pair("({} {} {})".format(alo, x.op, blo), "({} {} {})".format(ahi, x.op, bhi))
                    if isinstance(x, ex.Neg):
                        va = val(x.a)
                        if va[0] == "c":
                            return negc(va)
                        lo, hi = lanes(va)
                        return new_pair("(-{})".format(lo), "(-{})".format(hi))
                    if isinstance(x, ex.Cmp):
                        va, vb = val(x.a), val(x.b)
                        if va[0] == "c" and vb[0] == "c":
                            return ("cb", "({} {} {})".format(va[1], x.op, vb[1]))
                        (alo, ahi), (blo, bhi) = lanes(va), lanes(vb)
                        n = self.tmp()
                        e("const bool {n}l = ({} {op} {}), {n}h = ({} {op} {});".format(
                            alo, blo, ahi, bhi, n=n, op=x.op), 3)
                        return ("b", n + "l", n + "h")
                    if isinstance(x, ex.Logic):
                        vs = [val(y) for y in x.args]
                        if x.op == "not":
                            lo, hi = lanes(vs[0])
                            if vs[0][0] == "cb":
                                return ("cb", "(!{})".format(lo))
                            return ("b", "(!{})".format(lo), "(!{})".format(hi))
                        j = " && " if x.op == "and" else " || "
                        if all(v[0] == "cb" for v in vs):
                            return ("cb", "(" + j.join(v[1] for v in vs) + ")")
                        return ("b", "(" + j.join(lanes(v)[0] for v in vs) + ")",
                                "(" + j.join(lanes(v)[1] for v in vs) + ")")
                    if isinstance(x, ex.Select):
                        vc, va, vb = val(x.cond), val(x.a), val(x.b)
                        (clo, chi), (alo, ahi), (blo, bhi) = lanes(vc), lanes(va), lanes(vb)
                        lo = "({} ? {} : {})".format(clo, alo, blo)
                        hi = "({} ? {} : {})".format(chi, ahi, bhi)
                        if va[0] in ("b", "cb") and vb[0] in ("b", "cb"):
                            return ("b", lo, hi)
                        if vc[0] == "cb" and va[0] == "c" and vb[0] == "c":
                            return ("c", lo)
                        return new_pair(lo, hi)
                    if isinstance(x, ex.Call):
                        vs = [val(y) for y in x.args]
                        if all(v[0] == "c" for v in vs):
                            return ("c", "{}({})".format(math_fn[x.fn], ", ".join(v[1] for v in vs)))
                        return new_pair("{}({})".format(math_fn[x.fn], ", ".join(lanes(v)[0] for v in vs)),
                                        "{}({})".format(math_fn[x.fn], ", ".join(lanes(v)[1] for v in vs)))
                    raise TypeError(type(x))

                def fma(x):
                    """a*b + c, c + a*b, a*b - c (c uniform), c - a*b (a or b uniform) as one FFMA2."""
                    for mul, other, mul_first in ((x.a, x.b, True), (x.b, x.a, False)):
                        if not (isinstance(mul, ex.Bin) and mul.op == "*"):
                            continue
                        if isinstance(other, ex.Bin) and other.op == "*" and not mul_first:
                            continue
                        ma, mb, vo = val(mul.a), val(mul.b), val(other)
                        if not packable(ma, mb, vo) or (ma[0] == "c" and mb[0] == "c"):
                            # evaluate the conventional way from the values already emitted
                            vm = (("c", "({} * {})".format(ma[1], mb[1])) if ma[0] == "c" and mb[0] == "c" else
                                  packed("sf_mul2", ma, mb) if packable(ma, mb) else
                                  new_pair("({} * {})".format(lanes(ma)[0], lanes(mb)[0]),
                                           "({} * {})".format(lanes(ma)[1], lanes(mb)[1])))
                            va, vb = (vm, vo) if mul_first else (vo, vm)
                            if va[0] == "c" and vb[0] == "c":
                                return ("c", "({} {} {})".format(va[1], x.op, vb[1]))
                            if packable(va, vb):
                                return packed("sf_add2" if x.op == "+" else "sf_sub2", va, vb)
                            (alo, ahi), (blo, bhi) = lanes(va), lanes(vb)
                            return new_pair("({} {} {})".format(alo, x.op, blo), "({} {} {})".format(ahi, x.op, bhi))
                        if x.op == "+":
                            return packed("sf_fma2", ma, mb, vo)
                        if mul_first:                       # a*b - c
                            if vo[0] == "c":
                                return packed("sf_fma2", ma, mb, negc(vo))
                            return packed("sf_sub2", packed("sf_mul2", ma, mb), vo)
                        if ma[0] == "c":                    # c - a*b
                            return packed("sf_fma2", negc(ma), mb, vo)
                        if mb[0] == "c":
                            return packed("sf_fma2", ma, negc(mb), vo)
                        return packed("sf_sub2", vo, packed("sf_mul2", ma, mb))
                    return None

                for s in op.statements:
                    local[s.target] = val(s.value)
                target = op.name if op.name in local else op.statements[-1].target
                v = local[target]
                dst = "nv[{}][{}]".format(r, h)
                if v[0] == "p":
                    e("{} = {};".format(dst, v[1]), 3)
                elif v[0] == "c":
                    e("{0} = make_float2({1}, {1});".format(dst, v[1]), 3)
                else:
                    lo, hi = lanes(v)
                    e("{d}.x = {lo}; {d}.y = {hi};".format(d=dst, lo=lo, hi=hi), 3)

    def _emit_shifts(self, src, vec, tag, rr, age, nl, nr, u):
        """Left/right neighbour cells of an owned row: warp shuffles, plus the column ring at warp
        edges when several warps share a row."""
        g, e, T, V = self.geo, self.emit, self.T, self.geo.V
        f = self.fid[src.name]
        if nl:
            e("{T} l_{tag}[{n}];".format(T=T, tag=tag, n=nl), 3)
            for q in range(nl):
                e("l_{tag}[{q}] = __shfl_up_sync(0xffffffffu, {c}, 1, {w});".format(
                    tag=tag, q=q, c=self.cellref(vec, V - nl + q), w=g.KS), 3)
        if nr:
            e("{T} g_{tag}[{n}];".format(T=T, tag=tag, n=nr), 3)
            for q in range(nr):
                e("g_{tag}[{q}] = __shfl_down_sync(0xffffffffu, {c}, 1, {w});".format(
                    tag=tag, q=q, c=self.cellref(vec, q), w=g.KS), 3)
        if src.col_ring and (nl or nr):
            slot = self.ring_slot("xc_" + f, src.col_ring, age, u)
            n = src.col_reach
            sz = g.R * n
            # only the lane at a warp edge that has a neighbouring warp reads the ring word (predicated load)
            if nl:
                base = "xcol_{f} + ((({slot} * {WR} + wr) * {WC} + max(wc - 1, 0)) * 2 + 1) * {sz} + {o}".format(
                    f=f, slot=slot, WR=g.WR, WC=g.WC, sz=sz, o=rr * n)
                for q in range(nl):
                    e("if (lane == 0 && wc > 0) l_{tag}[{q}] = ({base})[{c}];".format(
                        tag=tag, q=q, base=base, c=n - nl + q), 3)
            if nr:
                base = "xcol_{f} + ((({slot} * {WR} + wr) * {WC} + min(wc + 1, {last})) * 2) * {sz} + {o}".format(
                    f=f, slot=slot, WR=g.WR, WC=g.WC, last=g.WC - 1, sz=sz, o=rr * n)
                for q in range(nr):
                    e("if (lane == 31 && wc < {lastw}) g_{tag}[{q}] = ({base})[{c}];".format(
                        tag=tag, q=q, base=base, c=q, lastw=g.WC - 1), 3)

    def _var(self, name, local, op):
        if name in local:
            return local[name]
        if name in self.specialize:
            return value_literal(self.specialize[name], self.ct)
        if name in self.program.constants:
            return value_literal(self.program.constants[name]["value"], self.ct)
        if name in self.sc_name:
            return "({}){}".format(self.T, self.sc_name[name])
        raise NameError("Unknown name {} in operator {}".format(name, op.name))


# ---------------------------------------------------------------------------------- planning


def register_limit(threads):
    """Registers per thread a single resident CTA of ``threads`` threads can have: each of the four
    SM sub-partitions holds 16384 registers and ceil(warps / 4) of the CTA's warps."""
    warps = -(-threads // 32)
    return min(255, (16384 // (-(-warps // 4) * 32)) // 8 * 8)


def _vector_width(program, dtype, options=None):
    """Consecutive cells a thread owns along the innermost dimension: 16 bytes by default (one
    128-bit shared-memory load / global store per row); ``options.vector`` asks for a longer run."""
    v = 16 // dtype.bytes
    want = getattr(options, "vector", 0) or v
    if want > v and want % v == 0 and program.shape[-1] % (want * 32) == 0:
        v = want
    if program.shape[-1] % v == 0 or unaligned_rows(program, dtype, options):
        return v                    # (unaligned rows: the last vector of a row is ragged)
    return None


def unaligned_rows(program, dtype, options):
    """True when a group of ``dtype`` fields is streamed in unaligned-row mode (``PlanOptions.unaligned``): its
    innermost rows are not a multiple of 16 bytes long, and the plan allows it (not in slab mode)."""
    return bool(getattr(options, "unaligned", 0) and not getattr(options, "peer_push", False)
                and (program.shape[-1] * dtype.bytes) % 16 != 0)


def candidate_geometries(program, ops, options):
    """(R, row groups, column warps, threads per row) candidates for a group, most specific first.
    Explicit ``rows_per_thread`` / ``warps`` options restrict the list."""
    dtype = ops[0].data_type
    ndim = len(program.shape)
    V = _vector_width(program, dtype, options)
    if V is None:
        return V, []
    nk = program.shape[-1]
    out = []
    if ndim == 3:
        rows = [options.rows_per_thread] if options.rows_per_thread else [4, 5, 3, 2, 1]
        warps = [options.warps] if options.warps else [16, 12, 10, 8]
        for R in rows:
            for w in warps:
                out.append((R, w, 1, 32))
        if nk >= 32 * V:
            # rows of 16 threads, two row groups per warp: a squarer tile (less halo to recompute)
            for R in rows:
                for w in warps:
                    out.append((R, 2 * w, 1, 16))
        if nk < 32 * V and nk // V <= 64:
            # narrow innermost dimension: one row of nk/V threads, several row groups per warp
            ks = nk // V
            for R in rows:
                for groups in ([options.warps * 32 // ks] if options.warps else [32, 24, 16, 12, 8]):
                    if groups and (groups * ks) % 32 == 0 and groups * ks <= 768:
                        out.append((R, groups, 1, ks))
    else:
        # 2-D rows: the warps of a CTA sit side by side; small CTAs (2-4 warps) let several independent
        # CTAs share an SM, each with its own barrier and TMA ring
        for w in ([options.warps] if options.warps else [1, 2, 4, 8, 16]):
            out.append((1, 1, w, 32))
    ks = getattr(options, "threads_per_row", 0)
    if ks:
        out = [c for c in out if c[3] == ks]
    return V, out


# Cost model of the planner (seconds), calibrated on B200 (profiles/r01_sweeps.txt): a streamed pass
# costs max(HBM time of its algorithmic bytes, time to compute its cells incl. the redundant halo
# cells).  The compute rate depends on the rows a thread owns (fewer rows = more exchange traffic per
# cell through shared memory, the co-limiter of the fused kernels) and collapses when the register
# windows do not fit the register file of the chosen CTA size.
def _measured_hbm_rate():
    """Bytes per second a streaming kernel can expect: 0.95 of the copy bandwidth the driver measured on this
    pool (``MEASURED_PEAKS.json``; the hdiff pass sustains 0.97 of it), 6.1 TB/s when that file is absent."""
    try:
        import json
        path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")
        with open(path) as f:
            return 0.95e9 * float(json.load(f)["hbm_gbs"])
    except Exception:
        return 6.1e12


HBM_BYTES_PER_S = _measured_hbm_rate()
# computed cell updates per second (halo cells included) of a fused 3-D pass at R = 4 rows per thread and 8
# warps, by element size: float32 from the Jacobi-3D chain (1024^3, depth 4, 64x64 tile: 4.25 ms per step)
UPDATES_PER_S = {4: 2.85e12, 8: 0.95e12}
UPDATES_PER_S_2D = {4: 2.7e12, 8: 1.95e12}  # 2-D rows, 8-warp CTAs (float64: 16 operators in 9.07 ms, r01c)
# rate relative to R = 4 (measured on the same chain, each at the largest CTA its registers allow: R = 3 x 12
# warps 3.84 ms on a 72x64 tile, R = 2 x 16 warps 4.76 ms; fewer rows = more exchange traffic per cell, but
# more warps per scheduler to hide it)
ROW_FACTOR = {1: 0.45, 2: 0.89, 3: 1.05, 4: 1.0, 5: 1.0}
# 2-D rows: compute rate of a CTA of w warps relative to 8 warps, measured on the float64 chain
# (profiles/r01c_sweep_config3_small_ctas.txt, re-measured with the short chunks of round 2,
# profiles/r02_sweep_sync_config3.txt: 1 / 2 / 4 warps 6.60 / 7.50 / 7.44 ms; tile efficiency factored out):
# independent small CTAs that start at different times hide each other's barrier and exchange latency
SMALL_CTA_FACTOR_2D = {1: 1.39, 2: 1.14, 4: 1.11}
PREFETCH_FACTOR = {5: 0.97}                 # 3-D passes: modelled time with the TMA ring 5 planes ahead instead of 2
GENERAL_EFFICIENCY = 0.84                   # fraction of HBM bandwidth the one-operator kernel reaches
LAUNCH_LATENCY = 2.4e-6                     # a small kernel behind another on one stream (8 launches of 32^3: 19.4 us)
# one streamed plane step per fused operator when nothing else limits it: barrier + exchange of a CTA, which
# grows with its warps (12-warp 3-D CTAs: 9 steps of 4 operators on 32^3 in 12 us; 2-warp 2-D CTAs: 0.05 us)
STEP_LATENCY_PER_WARP = 0.018e-6
STEP_LATENCY_3D = 0.2e-6
STREAM_SETUP = 3.0e-6                       # prologue of a streamed kernel before its first plane


def _tile_efficiency(ana, geo):
    if ana.ndim == 3:
        return (geo.BJ * geo.BK) / float(geo.TR * geo.TC)
    return geo.BK / float(geo.TC)


def modelled_time(program, ops, ana, geo):
    fields = program.fields
    eff = _tile_efficiency(ana, geo)
    # every tile loads its halo too: the memory system moves the inputs 1 / (tile efficiency) times (the
    # neighbouring tile's copy mostly comes from L2, but it still has to come)
    nbytes = sum(fields[i.name].nbytes for i in ana.ext_fields) / eff
    nbytes += sum(fields[i.name].nbytes for i in ana.fields.values() if i.stored)
    # tiles that stick out of the domain compute cells nobody stores (80 rows under 32-row tiles = 3 tiles)
    nk = program.shape[-1]
    used = nk / float(-(-nk // geo.BK) * geo.BK)
    if ana.ndim == 3:
        nj = program.shape[-2]
        used *= nj / float(-(-nj // geo.BJ) * geo.BJ)
    # a pass bound by HBM needs enough warps in flight to keep the memory system busy (hdiff: 5 warps per
    # SM reach 0.79 of what 15 warps do)
    t_mem = nbytes / (HBM_BYTES_PER_S * min(1.0, 0.7 + 0.02 * (geo.NT // 32) * resident_estimate(geo)))
    table = UPDATES_PER_S if ana.ndim == 3 else UPDATES_PER_S_2D
    rate = float(os.environ.get("SFB200_RATE_F{}".format(ana.dtype.bytes * 8), table[ana.dtype.bytes]))
    rate *= ROW_FACTOR.get(geo.R, 1.0) if ana.ndim == 3 else SMALL_CTA_FACTOR_2D.get(geo.NT // 32, 1.0)
    t_cmp = program.cells * len(ops) / (eff * used) / rate
    # latency floor: a CTA streams its planes one after the other, warm-up planes included, however few
    # cells a plane has (what a 32^3 grid costs: 9 steps of 4 fused operators measured 12 us)
    tiles = -(-nk // geo.BK) * (-(-program.shape[-2] // geo.BJ) if ana.ndim == 3 else 1)
    slots = SM_COUNT * resident_estimate(geo)
    overhead = ana.t_end_offset() - ana.t_begin_offset()
    n_stream = program.shape[0]
    steps = overhead + (-(-n_stream * tiles // slots) if tiles >= slots else -(-n_stream // (slots // tiles)))
    per_op_step = STEP_LATENCY_PER_WARP * (geo.NT // 32)
    if ana.ndim == 3:
        # ... and however few warps: TMA wait, ring loads, the dependent arithmetic and the barrier of one
        # operator on one plane take ~0.2 us, and a streamed kernel spends ~3 us before its first plane
        # (barriers, descriptors, the first TMA round trip): 2-warp CTAs on 32^3 run 9 steps of 4 operators
        # in 14.7 us (ncu), eight one-operator launches of the same program take 24 us in total
        per_op_step = max(per_op_step, STEP_LATENCY_3D)
    t_lat = steps * per_op_step * len(ops)
    return max(t_mem, t_cmp, t_lat) + LAUNCH_LATENCY + STREAM_SETUP


def choose_geometry(program, ops, options):
    """Pick (V, R, warps, prefetch) for a candidate group -- the admissible geometry with the lowest
    modelled pass time -- or return None when the group cannot stream."""
    import copy
    trials = [options]
    if len(program.shape) == 2 and not getattr(options, "vector", 0):
        # 2-D rows: 32 bytes per thread first (half the shuffles and ring words per cell; measured
        # 1.27x faster than 16 bytes on the float64 chain, profiles/r01_sweep_sync_prefetch.txt)
        wide = copy.copy(options)
        wide.vector = 32 // ops[0].data_type.bytes
        trials = [wide, options]
    best = None
    # (the cost model prices a pass over unaligned rows like an aligned one)
    unaligned = unaligned_rows(program, ops[0].data_type, options)
    for opts in trials:
        try:
            V, candidates = candidate_geometries(program, ops, opts)
            if V is None:
                continue
            # TMA ring depth - 1: 2 planes ahead by default; 2-D rows are small (a ring of 6 fits many
            # times) and measured fastest with 5 (profiles/r01_sweep_sync_prefetch.txt)
            # 3-D tiles: both ring depths compete -- 5 planes ahead is worth ~3 % (ring depth 6 = the unroll
            # factor; Jacobi-3D 4.18 -> 4.03 ms) unless the deeper ring costs the tile rows its shared memory
            # would have held (hdiff: 48 -> 32 rows, 0.162 -> 0.180 ms)
            prefetches = [opts.prefetch] if opts.prefetch else ([5] if len(program.shape) == 2 else [5, 2])
            explicit = bool(opts.rows_per_thread and opts.warps)
            for (R, WR, WC, KS) in candidates:
                for prefetch in prefetches:
                    try:
                        ana = GroupAnalysis(program, ops, exchange_cols=(WC > 1))
                        sync = getattr(opts, "sync", "") or DEFAULT_SYNC
                        direct = bool(getattr(opts, "direct", 0))
                        tmem = int(getattr(opts, "tmem", 0) or 0)
                        geo = Geometry(ana, V, R, WR, WC, prefetch, KS, sync, direct=direct, tmem=bool(tmem),
                                       unaligned=unaligned)
                        if geo.tmem and tmem < 2 and ana.register_estimate(R, V) < register_limit(geo.NT):
                            # the windows fit the registers: nothing to park (tmem = 2 parks all the same, so
                            # that the tensor-memory code of passes far from their register limit can be tested)
                            geo = Geometry(ana, V, R, WR, WC, prefetch, KS, sync, direct=direct, unaligned=unaligned)
                        elif geo.tmem and not getattr(opts, "sync", ""):
                            # a pass at its register limit spends what the parked planes free on per-field
                            # mbarriers instead of the CTA barrier (Jacobi-3D 1024^3: 3.69 vs 3.84 ms; parked
                            # planes under the CTA barrier alone: 4.04 ms, profiles/r03_sweep_tmem_config1.txt)
                            geo = Geometry(ana, V, R, WR, WC, prefetch, KS, "flags", direct=direct, tmem=True,
                                           unaligned=unaligned)
                    except NotStreamable:
                        break
                    if geo.smem > SMEM_LIMIT:
                        continue
                    if not explicit and ana.register_estimate(R, V, geo.tmem) > register_limit(geo.NT) + REG_SLACK:
                        continue
                    t = modelled_time(program, ops, ana, geo)
                    if len(program.shape) == 3 and len(prefetches) > 1:
                        t *= PREFETCH_FACTOR.get(prefetch, 1.0)
                    if best is None or t < best[0] * (1 - 1e-6):
                        best = (t, ana, geo)
        except NotStreamable:
            continue
    if best is None:
        return None
    return best[1], best[2]


def group_cost(program, ops, options):
    """Estimated time of one streamed pass over ``ops`` (None if the group cannot stream)."""
    chosen = choose_geometry(program, ops, options)
    if chosen is None:
        return None
    ana, geo = chosen
    return modelled_time(program, ops, ana, geo)


def general_cost(program, op):
    fields = program.fields
    nbytes = fields[op.name].nbytes + sum(fields[f].nbytes for f in op.accesses)
    return nbytes / (HBM_BYTES_PER_S * GENERAL_EFFICIENCY) + LAUNCH_LATENCY


def partition(program: StencilProgram, options):
    """Cut the topologically ordered operators into passes minimising the modelled run time
    (dynamic programme over contiguous groups of at most ``max_depth`` operators)."""
    ops = list(program.ops)
    n = len(ops)
    if options.max_depth:
        # an explicit depth is a request, not a bound: the longest streamable run of at most that
        # many operators, repeatedly (what the tuner and the SFB200_MAX_DEPTH sweeps ask for)
        groups, start = [], 0
        while start < n:
            for depth in range(min(options.max_depth, n - start), 0, -1):
                group = ops[start:start + depth]
                if group_cost(program, group, options) is not None:
                    groups.append(("streamed", group))
                    break
                if depth == 1:
                    groups.append(("general", group))
            start += len(groups[-1][1])
        return groups
    max_depth = 8
    best = [0.0] + [None] * n          # best[k]: cost of the first k operators
    choice = [None] * (n + 1)
    cache = {}
    for end in range(1, n + 1):
        for start in range(max(0, end - max_depth), end):
            group = ops[start:end]
            # structurally identical chain segments (Jacobi chains) share one estimate
            chain = _chain_like(group)
            # (what decides streamability and cost: taps, boundary handling, result type -- and the
            # type and dimensionality of the field the chain starts from)
            key = None
            if chain:
                src = program.fields[next(iter(group[0].accesses))]
                key = (src.data_type.name, tuple(src.dims)) + tuple(
                    (repr([op.offsets3(f) for f in op.accesses]),
                     repr(sorted(op.boundary_conditions.items(), key=repr)[0][1:] if op.boundary_conditions else ""),
                     op.data_type.name, tuple(sorted(op.scalars))) for op in group)
            if chain and key in cache:
                cost = cache[key]
            else:
                cost = group_cost(program, group, options)
                if chain:
                    cache[key] = cost
            family = "streamed"
            if len(group) == 1:
                # a single operator may also be cheaper as a one-operator kernel (tiny grids: no warm-up planes)
                alone = general_cost(program, group[0])
                if cost is None or alone < cost:
                    cost, family = alone, "general"
            elif cost is None:
                continue
            if best[start] is None:
                continue
            total = best[start] + cost
            if best[end] is None or total < best[end] - 1e-12:
                best[end] = total
                choice[end] = (start, family)
    groups = []
    end = n
    while end > 0:
        start, family = choice[end]
        groups.append((family, ops[start:end]))
        end = start
    groups.reverse()
    return groups


def _chain_like(group):
    """True when every operator reads exactly one array field: the previous operator's result
    (or the group's single input) -- the case where cost estimates can be shared."""
    prev = None
    for op in group:
        if len(op.accesses) != 1:
            return False
        (field,) = op.accesses.keys()
        if prev is not None and field != prev:
            return False
        prev = op.name
    return True


def choose_chunk(n_stream, tiles, overhead, sms=148, max_len=None):
    """Planes per CTA along the streamed dimension: balance wave quantisation against the
    redundant warm-up planes every chunk recomputes.  ``max_len``: longest chunk considered (2-D rows: many
    short CTAs run measurably faster than few long ones, see lower_group)."""
    best = None
    for chunks in range(1, 65 * max(1, sms // 148)):
        ci = -(-n_stream // chunks)
        if max_len and ci > max_len and chunks + 1 < 65 * max(1, sms // 148):
            continue
        blocks = tiles * (-(-n_stream // ci))
        waves = -(-blocks // sms)
        cost = waves * (ci + overhead)
        if best is None or cost < best[0]:
            best = (cost, ci)
    return best[1]


def schedule_work(n_tiles, n_planes, slots, overhead, edge_tiles=None):
    """Work items of a streamed pass for its persistent CTAs: ``[(tile, p_begin, p_end), ...]``, planes
    relative to the first plane of the slab, in the order the CTAs fetch them (CTA b starts with item
    b, every CTA then takes the next unclaimed one).

    Two things make a pass fast.  (1) The CTAs running at any moment should work on *adjacent tiles at
    (nearly) the same planes*: the halo two neighbouring tiles both read then comes from L2 instead of
    HBM and DRAM pages are used whole -- cutting the (tile, plane) space into ``slots`` equal linear
    shares, every CTA somewhere else, was measured 43 % slower on the Jacobi-3D chain (DESIGN 3.2).
    (2) Every CTA should stop at the same time although tiles differ in speed (domain-edge tiles run
    the boundary code in every step).  So the list is

    * whole tiles first, in waves of ``slots`` neighbours that stream in lockstep and pay the warm-up
      planes once per tile -- as many waves as leave enough other work to even out the differences the
      whole tiles produce (``EDGE_SLOWDOWN`` per wave);
    * then the remaining tiles in rounds of plane ranges that halve from round to round (factoring
      self-scheduling): each round hands about half of what is left to ``slots`` items of equal length,
      tile-minor so that the CTAs of a round hold adjacent tiles of one range; the last items are short
      (a few times the warm-up), which bounds how far apart the CTAs finish."""
    mode = os.environ.get("SFB200_SCHED", SCHED_DEFAULT)
    if mode in ("lpt", "rows") and edge_tiles is not None and n_tiles >= 2 * slots:
        return _schedule_longest_first(n_tiles, n_planes, slots, overhead, edge_tiles, by_rows=(mode == "rows"))
    whole = int((n_tiles / float(slots)) / (1.0 + EDGE_SLOWDOWN)) * slots
    items = [(t, 0, n_planes) for t in range(whole)]
    tiles = n_tiles - whole
    if tiles:
        pieces = max(1, int(round(slots / float(tiles))))          # ranges per tile and round
        floor_ = max(4 * overhead, 16)                               # shortest range worth a warm-up
        pos = 0
        share = 1.0 / (1.0 + EDGE_SLOWDOWN) if not whole else 0.5    # first round: all but the slack
        while pos < n_planes:
            rest = n_planes - pos
            size = max(floor_, -(-int(rest * share) // pieces))
            share = 0.5
            if rest - pieces * size < floor_:                        # last round: no stub shorter than the floor
                k = max(1, min(pieces, rest // floor_))
                size = -(-rest // k)
            else:
                k = pieces
            for c in range(k):
                b, e_ = pos + c * size, min(n_planes, pos + (c + 1) * size)
                if b < e_:
                    items.extend((whole + t, b, e_) for t in range(tiles))
            pos += k * size
    # few tiles, short slab: plain equal ranges sized for whole waves use the slots better
    ctas = min(slots, len(items))
    steps = [e_ - b + overhead for (_, b, e_) in items]
    cost = max(sum(steps) / float(ctas), max(steps)) + min(steps)
    ci = choose_chunk(n_planes, n_tiles, overhead, sms=slots)
    nchunk = -(-n_planes // ci)
    if -(-n_tiles * nchunk // slots) * (ci + overhead) < cost:
        return [(t, c * ci, min(n_planes, (c + 1) * ci)) for c in range(nchunk) for t in range(n_tiles)]
    return items


def _schedule_longest_first(n_tiles, n_planes, slots, overhead, edge_tiles, by_rows=False):
    """Alternative list for passes with at least two tiles per slot: every full wave of tiles streams whole
    (one warm-up per tile), the *domain-edge tiles first* -- they are the slow ones, and the CTAs that drew
    them simply fetch their next tile later (longest-processing-time-first) -- and only the tiles that do not
    fill a wave are cut into halving plane ranges that even out the finish."""
    edge = [t for t in range(n_tiles) if t in edge_tiles]
    inner = [t for t in range(n_tiles) if t not in edge_tiles]
    order = edge + inner
    if by_rows:
        # (experiment) keep the tiles in index order -- whole tile rows side by side, better halo sharing in
        # L2 -- and only bring the runs of edge tiles at both ends of the index range to the front
        first_inner = next((t for t in range(n_tiles) if t not in edge_tiles), 0)
        last_inner = max([t for t in range(n_tiles) if t not in edge_tiles] + [0])
        head = list(range(0, first_inner)) + list(range(last_inner + 1, n_tiles))
        order = head + list(range(first_inner, last_inner + 1))
    whole = (n_tiles // slots) * slots
    items = [(t, 0, n_planes) for t in order[:whole]]
    rest = order[whole:]
    if rest:
        pieces = max(1, slots // len(rest))
        floor_ = max(2 * overhead, 16)
        pos, share = 0, 0.75
        while pos < n_planes:
            left = n_planes - pos
            size = max(floor_, -(-int(left * share) // pieces))
            share = 0.5
            if left - pieces * size < floor_:
                k = max(1, min(pieces, left // floor_))
                size = -(-left // k)
            else:
                k = pieces
            for c in range(k):
                b, e_ = pos + c * size, min(n_planes, pos + (c + 1) * size)
                if b < e_:
                    items.extend((t, b, e_) for t in rest)
            pos += k * size
    return items


def pack_work_table(items):
    """int32 table the kernel reads and updates: [next-item counter, finished-CTA counter, number of
    items], then 3 ints per item.  Both counters are zero between launches (the last CTA resets them)."""
    flat = [0, 0, len(items)]
    for item in items:
        flat.extend(item)
    return flat


def resident_estimate(geo):
    """CTAs of a streamed kernel an SM holds at once (the executor asks the driver for the exact figure
    once the function is loaded): registers at 255 per thread under __launch_bounds__(NT, 1), shared
    memory, the 32-CTA limit."""
    return max(1, min(65536 // (256 * geo.NT), SMEM_LIMIT // max(geo.smem, 1), 32))


def lower_group(lowered: LoweredProgram, ops: List[StencilOp], options, specialize=None):
    program = lowered.program
    chosen = choose_geometry(program, ops, options)
    if chosen is None:
        raise NotStreamable("group cannot stream")
    ana, geo = chosen
    # the cell copies of unaligned rows index the whole field (all NS planes, zero-fill past its ends): a slab buffer,
    # which holds only some planes, would be read past its end -- unaligned_rows() keeps the mode out of slab mode
    assert not (geo.unaligned and getattr(options, "peer_push", False))
    gen = StreamKernelGen(program, ops, ana, geo, specialize, peer_push=bool(getattr(options, "peer_push", 0)))
    name, src, args = gen.generate()
    if name not in lowered.kernels:
        lowered.kernels[name] = KernelSpec(name, src, (geo.NT, 1, 1), "streamed",
                                           prelude=UNALIGNED_PRELUDE if geo.unaligned else "")
    NI, NJ, NK = program.shape3
    n_stream = program.shape[0]
    gx = -(-NK // geo.BK)
    gy = -(-NJ // geo.BJ) if ana.ndim == 3 else 1
    overhead = ana.t_end_offset() - ana.t_begin_offset()
    # CTAs of this kernel an SM holds at once: small CTAs (1-4 warps, the warp-private 2-D tiles) share an
    # SM, limited by the register file (ptxas may use 255 registers under __launch_bounds__(NT, 1)),
    # shared memory and the 32-CTA limit; the chunking must fill all of those slots
    resident = resident_estimate(geo)

    def chunk_for(b, e_):
        if options.chunk:
            return options.chunk
        # 2-D rows: chunks of at most 32 x the warm-up rows.  The float64 chain runs 4.7 % faster with 68-79
        # chunks of 416-482 rows (16-18 "waves" of CTAs) than with the 30 chunks of 1093 rows that minimise
        # waves x (rows + warm-up): 7.79 -> 7.40-7.45 ms (profiles/r02_sweep_sync_config3.txt); CTAs that start
        # at different times keep the four CTAs of an SM out of phase with each other
        cap = 32 * overhead if ana.ndim == 2 else None
        return choose_chunk(max(1, e_ - b), gx * gy, overhead, sms=SM_COUNT * resident, max_len=cap)

    def work_items(b, e_, resident_ctas=None):
        """Work items of the persistent CTAs for planes [b, e_): one CTA per slot the device really
        offers (``resident_ctas`` = occupancy of the loaded function x SMs, supplied by the executor;
        the estimate otherwise)."""
        slots = resident_ctas or SM_COUNT * resident
        # tiles with cells outside the domain run the boundary code in every step
        edge = set()
        for t in range(gx * gy):
            kx, jy = t % gx, t // gx
            k0 = kx * geo.BK - geo.HK0
            if k0 < 0 or k0 + geo.TC > NK:
                edge.add(t)
            if ana.ndim == 3:
                j0 = jy * geo.BJ - geo.HJ0
                if j0 < 0 or j0 + geo.TR > NJ:
                    edge.add(t)
        return schedule_work(gx * gy, max(1, e_ - b), slots, overhead, edge_tiles=edge)

    def work_table(b, e_, resident_ctas=None):
        return pack_work_table(work_items(b, e_, resident_ctas))

    def grid(b, e_, resident_ctas=None):
        if gen.persistent:
            slots = resident_ctas or SM_COUNT * resident
            return (min(slots, len(work_items(b, e_, resident_ctas))), 1, 1)
        ci = chunk_for(b, e_)
        return (gx, gy, max(1, -(-(e_ - b) // ci)))

    stored = [i.name for i in ana.fields.values() if i.stored]
    reads = [i.name for i in ana.ext_fields] + list(ana.aux)
    reach = {i.name: (i.back, i.fwd) for i in ana.ext_fields}
    reach.update({name: tuple(r) for name, r in ana.aux_reach.items()})
    launch = LaunchSpec(kernel=name, grid_fn=grid, block=(geo.NT, 1, 1), smem=geo.smem, args=args,
                        ops=[op.name for op in ops], reads=reads, writes=stored,
                        cells_per_unit=program.cells * len(ops), family="streamed",
                        info={"V": geo.V, "R": geo.R, "warps": [geo.WR, geo.WC], "threads_per_row": geo.KS,
                              "tile": [geo.TR, geo.TC],
                              "block_out": [geo.BJ, geo.BK], "halo": [geo.HJ0, geo.HJ1, geo.HK0, geo.HK1],
                              "prefetch": geo.P, "persistent": gen.persistent, "peer_push": gen.peer_push,
                              "tiles": gx * gy, "sync": "pair" if geo.pair else ("halves" if geo.halves else ("flags" if gen.flags else "cta")), "direct": sorted(geo.direct), "unroll": gen.U, "packed": gen.G == 2, "halo_skip": [gen.rotate_rows, gen.skip_warps, gen.skip_from], "lags": {n: i.lag for n, i in ana.fields.items()},
                              "windows": {n: i.window for n, i in ana.fields.items() if i.consumed},
                              "window_registers": ana.window_registers(geo.R, geo.V),
                              "register_estimate": ana.register_estimate(geo.R, geo.V, geo.tmem),
                              "tmem": dict(ana.tmem_ages) if gen.tmem else {},
                              # where a step parks each of them: after operator k, -1 after the inputs, -2 first
                              "tmem_store": {f.name: k for k, fs in gen._tm_store_points(ops).items() for f in fs},
                              "stream_overhead_planes": overhead,
                              "back": max(i.back for i in ana.fields.values()),
                              "reach": reach,
                              "tile_efficiency": _tile_efficiency(ana, geo),
                              "fwd": ana.max_lag,
                              "chunk_fn": chunk_for, "work_fn": work_table, "work_items_fn": work_items})
    if geo.unaligned:
        launch.info["unaligned"] = True       # (recorded for the passes that run so only: other records stay as they were)
    lowered.launches.append(launch)
    lowered.uses_stream = True
    return launch
