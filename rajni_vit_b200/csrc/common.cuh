// Shared helpers for the sm_100a kernels.  Host side: errors, the launch path (launch_kernel, launch_checked,
// raise_smem_limit), the SM count and the TMA tensor-map builders.  Device side: mbarrier, TMA, cp.async, tcgen05/TMEM
// wrappers, warp reductions, vector loads and stores.  Inline PTX only — no CUTLASS.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <utility>

#include "../../include/rajni_b200.h"

namespace rajni {

// ------------------------------------------------------------------ host-side errors (runtime.cu)
void set_error(const char* fmt, ...);
const char* error_text();             // the calling thread's last message
uint64_t launches();
void count_launch(int n = 1);
int check_launch(const char* what);   // cudaGetLastError -> RAJNI_ECUDA

#define RAJNI_REQUIRE(cond, code, ...)            \
    do {                                          \
        if (!(cond)) {                            \
            ::rajni::set_error(__VA_ARGS__);      \
            return (code);                        \
        }                                         \
    } while (0)

// ------------------------------------------------------------------ programmatic dependent launch
// Every kernel of the path is launched with cudaLaunchAttributeProgrammaticStreamSerialization: it may start
// (set up shared memory, barriers, TMEM, descriptors) while its predecessor in the stream is still draining, and
// blocks in griddep_wait() until that predecessor has completed and flushed before it touches global memory.
// griddep_launch() lets the NEXT kernel do the same with respect to this one.
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

int current_device();    // runtime.cu: cudaGetDevice, 0 on error (indexes the per-device one-time flags below)
constexpr int kMaxDevices = 64;

template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                 int cluster_x, Args&&... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    int n = 0;
    if (cluster_x > 1) {
        attr[n].id = cudaLaunchAttributeClusterDimension;
        attr[n].val.clusterDim.x = cluster_x;
        attr[n].val.clusterDim.y = 1;
        attr[n].val.clusterDim.z = 1;
        ++n;
    }
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
    cfg.attrs = attr;
    cfg.numAttrs = n;
    return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

// launch_kernel, counted in rajni_launch_count() whether or not the launch call succeeds.  Returns RAJNI_OK, or
// RAJNI_ECUDA with `name` in the error text when the launch call or cudaGetLastError reports an error.
template <typename... KArgs, typename... Args>
inline int launch_checked(const char* name, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                          int cluster_x, Args&&... args) {
    const cudaError_t e = launch_kernel(kern, grid, block, smem, stream, cluster_x, std::forward<Args>(args)...);
    count_launch();
    RAJNI_REQUIRE(e == cudaSuccess, RAJNI_ECUDA, "%s: launch failed: %s", name, cudaGetErrorString(e));
    return check_launch(name);
}

// Raises `kern`'s dynamic shared-memory limit on the current device to `bytes`, calling the runtime only when `bytes`
// exceeds what `granted` (the caller's static record for this kernel, per device) says was already set there.
template <typename... KArgs>
inline int raise_smem_limit(const char* name, void (*kern)(KArgs...), int bytes, int (&granted)[kMaxDevices]) {
    int& g = granted[current_device()];
    if (bytes > g) {
        const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        RAJNI_REQUIRE(e == cudaSuccess, RAJNI_ECUDA, "%s: smem attribute (%d B): %s", name, bytes, cudaGetErrorString(e));
        g = bytes;
    }
    return RAJNI_OK;
}

// SM count of the current device, queried once per device (one process may drive several GPUs); 148 if the query fails.
inline int num_sms() {
    static int n_dev[kMaxDevices] = {};
    const int dev = current_device();
    int& n = n_dev[dev];
    if (!n) {
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

// ------------------------------------------------------------------ TMA tensor maps (gemm_tcgen05.cu)
// bf16, 128-byte swizzle, out-of-bounds elements read as zero.  Return 0 or RAJNI_ECUDA.
// 2-D row-major [rows, cols] with a leading dimension of ld_elems, box = box_rows x 64 columns (L2 promotion 256 B).
int make_tmap_bf16_2d(CUtensorMap* map, const void* base, long long rows, long long cols, long long ld_elems, int box_rows);
// 3-D densely packed [batch][rows][cols], box = box_rows x 64 columns of one batch entry: a box never crosses into the next
// entry's rows (stores are clipped there, loads zero-filled).  _box: no L2 promotion (stores); _ld: 256 B (loads).
int make_tmap_bf16_3d_box(CUtensorMap* map, const void* base, long long batch, long long rows, long long cols, int box_rows);
int make_tmap_bf16_3d_ld(CUtensorMap* map, const void* base, long long batch, long long rows, long long cols, int box_rows);

// ------------------------------------------------------------------ small device utils
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// streaming 16-byte load that does not pollute L1
__device__ __forceinline__ uint4 ld_stream16(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void prefetch_l2(const void* p) {
    asm volatile("prefetch.global.L2 [%0];" :: "l"(p));
}
__device__ __forceinline__ void st_stream16(void* p, const uint4& v) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ float2 bf16x2_to_float2(uint32_t u) {
    // bf16 -> fp32 is a 16-bit left shift
    return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u));
}
__device__ __forceinline__ uint32_t float2_to_bf16x2(float lo, float hi) {
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
}

// ---- packed fp32x2 arithmetic (sm_100: FFMA2 / FADD2 / FMUL2, two fp32 lanes per instruction)
__device__ __forceinline__ uint64_t f2pack(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void f2unpack(uint64_t v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
// 32-byte global accesses (sm_100: LDG.256 / STG.256)
__device__ __forceinline__ void ldg256_nc(const void* p, uint32_t (&v)[8]) {
    asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "l"(p));
}
// the same without .nc: for data the kernel itself also writes (a residual that aliases the output, model.py:55-59 in place)
__device__ __forceinline__ void ldg256(const void* p, uint32_t (&v)[8]) {
    asm volatile("ld.global.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "l"(p) : "memory");
}
__device__ __forceinline__ void stg256(void* p, const uint32_t (&v)[8]) {
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
// explicit shared-state-space store (a generic pointer into dynamic smem compiles to ST.E)
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" :: "r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
    float d;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                 :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}"
        :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}

// non-blocking probe: true once the phase with this parity has completed
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}

// ------------------------------------------------------------------ cp.async
// 16-byte global -> shared copy; the bytes past src_bytes (0 or 16) are zero-filled
__device__ __forceinline__ void cp_async16(uint32_t smem_dst, const void* gsrc, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" :: "r"(smem_dst), "l"(gsrc), "r"(src_bytes) : "memory");
}
// arrive on `bar` once every cp.async issued so far by this thread has landed
__device__ __forceinline__ void cp_async_arrive_noinc(uint64_t* bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" :: "r"(smem_u32(bar)) : "memory");
}

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
    asm volatile("prefetch.tensormap [%0];" :: "l"(tmap) : "memory");
}
// 2-D tile load: c0 = innermost (element) coordinate, c1 = row coordinate.
__device__ __forceinline__ void tma_load_2d(void* dst, const void* tmap, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        :: "r"(smem_u32(dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const void* tmap, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        :: "r"(smem_u32(dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// ---- 2-CTA (cta_group::2) variants: both CTAs of a pair load into their own smem but signal the
// LEADER CTA's mbarrier (a shared::cluster address obtained with mapa).
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t smem_addr, uint32_t cta_rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(cta_rank));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx_cluster(uint32_t bar_cluster_addr, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;"
                 :: "r"(bar_cluster_addr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" :: "r"(bar_cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_load_2d_cg2(void* dst, const void* tmap, uint32_t bar_cluster_addr, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        :: "r"(smem_u32(dst)), "l"(tmap), "r"(bar_cluster_addr), "r"(c0), "r"(c1) : "memory");
}
// generic-proxy smem writes -> visible to the async proxy (UMMA / TMA store)
__device__ __forceinline__ void fence_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// TMA store of one box (shared -> global), tracked by the issuing thread's bulk async-group
__device__ __forceinline__ void tma_store_3d(const void* tmap, uint32_t smem_src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                 :: "l"(tmap), "r"(smem_src), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all but the newest N groups of this thread have finished READING their shared-memory source
template <int N>
__device__ __forceinline__ void bulk_wait_group_read() { asm volatile("cp.async.bulk.wait_group.read %0;" :: "n"(N) : "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_group() { asm volatile("cp.async.bulk.wait_group %0;" :: "n"(N) : "memory"); }

// ------------------------------------------------------------------ tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {   // whole warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 :: "r"(smem_u32(dst_smem)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {     // whole warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t* dst_smem, uint32_t cols) {   // whole warp, in BOTH CTAs
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                 :: "r"(smem_u32(dst_smem)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" :: "r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; bf16 inputs, fp32 accumulate. One thread issues.
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                          uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// 2-CTA MMA: issued by the leader CTA only; A rows and B rows are split across the pair's smem,
// each CTA's TMEM receives its 128 accumulator rows.
__device__ __forceinline__ void umma_bf16_cg2(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                              uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// commit that arrives on the barrier at the same smem offset in every CTA of `cta_mask`
__device__ __forceinline__ void umma_commit_cg2(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 :: "r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}
// A operand from TMEM (lane = row, two bf16 per 32-bit column along K), B from smem.
__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc,
                                             uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        :: "r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive on an mbarrier once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                 :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets lane (base_lane+i).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr) : "memory");
}
// ---- 16-lane shapes: a warp addresses lanes [L, L+16) of its quadrant (L % 16 == 0); registers come in the mma
// accumulator-fragment layout (see attention_tc.cu).  16x256b.xR = 8R fp32 columns, 16x128b.xR = 4R 32-bit columns.
__device__ __forceinline__ void tmem_ld16x256_x2(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld16x256_x4(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld16x256_x8(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.16x256b.x8.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st16x128_x2(uint32_t taddr, const uint32_t (&v)[4]) {
    asm volatile("tcgen05.st.sync.aligned.16x128b.x2.b32 [%0], {%1,%2,%3,%4};"
                 :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]) : "memory");
}
__device__ __forceinline__ void tmem_st16x128_x4(uint32_t taddr, const uint32_t (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.16x128b.x4.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_st16x128_x8(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.16x128b.x8.b32 [%0], "
        "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
        :: "r"(taddr),
           "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
           "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
        :: "r"(taddr),
           "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
           "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
        :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
        : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
        "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
        :: "r"(taddr),
           "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
           "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
           "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
           "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
        : "memory");
}

// Shared-memory matrix descriptor for tcgen05.mma, 128-byte swizzle, bf16.
//   bits [0,14)  start address >> 4         bits [16,30) leading byte offset >> 4
//   bits [32,46) stride byte offset >> 4    bits [46,48) descriptor version (1 on sm_100)
//   bits [61,64) layout type (2 = SWIZZLE_128B)
// K-major tile  [rows][64 bf16]: rows are 128 B apart, 8-row groups 1024 B apart (SBO);
//                LBO is not used by the hardware for swizzled K-major layouts.
// MN-major tile [k][64 bf16]  : 64 MN-elements contiguous, 8 k-rows per 1024 B group (SBO);
//                LBO = distance between 64-element MN blocks.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3ffffu) >> 4);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3fffu) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3fffu) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}

// Instruction descriptor, kind::f16: bf16 x bf16 -> fp32.
//   [4,6) D format (1 = f32)  [7,10) A format (1 = bf16)  [10,13) B format (1 = bf16)
//   [15] A major (0 = K)      [16] B major (0 = K, 1 = MN)
//   [17,23) N >> 3            [24,29) M >> 4
__host__ __device__ __forceinline__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
    return (1u << 4) | (1u << 7) | (1u << 10) |
           (static_cast<uint32_t>(a_mn_major) << 15) | (static_cast<uint32_t>(b_mn_major) << 16) |
           (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

}  // namespace rajni
