// distrifuser_b200 -- fused all-reduce of the tensor-parallel path over NVLink peer memory.
// Replaces the blocking dist.all_reduce + bias add (+ residual add) of the reference's tensor-parallel modules:
// modules/tp/attention.py:159, feed_forward.py:77, resnet.py:189 and conv2d.py:52.
#include "common.cuh"

using namespace df;

namespace {

__device__ __forceinline__ void unpack8h(const int4& r, float f[8]) {
  const __half2* h = reinterpret_cast<const __half2*>(&r);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 t = __half22float2(h[j]);
    f[2 * j] = t.x;
    f[2 * j + 1] = t.y;
  }
}

__device__ __forceinline__ int4 pack8h(const float f[8]) {
  int4 r;
  __half2* h = reinterpret_cast<__half2*>(&r);
#pragma unroll
  for (int j = 0; j < 4; ++j) h[j] = __floats2half2_rn(f[2 * j], f[2 * j + 1]);
  return r;
}

constexpr int AR_THREADS = 256;
constexpr int AR_UNROLL = 4;   // 16-byte loads in flight per thread while pushing

// One-shot all-reduce.  Every member stores its partial into slot (ring, src = me) of every peer's arena with posted 16-byte
// stores, the last CTA to finish stamps the peers' flags (release, system scope) with the sequence number, then every member
// waits for all peers' flags and reduces the n slots of its OWN arena locally: fp32, sources in member order 0..n-1, then
// bias, then residual, rounded to fp16 once -- so every member writes the same bits.
// A member whose bit is clear in `contrib` pushes nothing (partial == nullptr) but still stamps its flags: the ring-reuse
// argument (utils.py, next to the BANK-REUSE INVARIANT) needs every member to pass every all-reduce.
__global__ void __launch_bounds__(AR_THREADS) allreduce_kernel(df_comm_t c, const __half* __restrict__ partial,
                                                               __half* __restrict__ out, uint64_t nvec, int C,
                                                               const __half* __restrict__ bias,
                                                               const __half* __restrict__ residual, uint32_t contrib,
                                                               int site, int nsites, uint64_t ring_off, uint64_t slot_bytes,
                                                               uint64_t flags_off, int ticket) {
  const int n = c.world, me = c.rank;
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  const uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t ring = 0;
  if (n > 1) {
    // sequence number = call epoch * sites + site: one captured graph replays forever (the clock advances on the device)
    const uint32_t seq = c.clock[0] * (uint32_t)nsites + (uint32_t)site;
    ring = seq % DF_AR_RING;
    const uint64_t my_slot = ring_off + (uint64_t)(ring * n + me) * slot_bytes;
    if (partial != nullptr) {
      uint64_t i = i0;
      for (; i + (AR_UNROLL - 1) * stride < nvec; i += AR_UNROLL * stride) {
        int4 v[AR_UNROLL];
#pragma unroll
        for (int u = 0; u < AR_UNROLL; ++u) v[u] = ld_nc_v4(partial + (i + u * stride) * 8);
        for (int p = 0; p < n; ++p) {
          if (p == me) continue;
          char* dst = (char*)c.base[p] + my_slot;
#pragma unroll
          for (int u = 0; u < AR_UNROLL; ++u) st_v4(dst + (i + u * stride) * 16, v[u]);
        }
      }
      for (; i < nvec; i += stride) {
        const int4 v = ld_nc_v4(partial + i * 8);
        for (int p = 0; p < n; ++p)
          if (p != me) st_v4((char*)c.base[p] + my_slot + i * 16, v);
      }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
      const uint32_t t = atomicAdd(&c.tickets[ticket], 1u);
      if (t == gridDim.x - 1) {
        __threadfence();
        c.tickets[ticket] = 0;  // the next all-reduce is stream-ordered after this kernel
        for (int p = 0; p < n; ++p)
          if (p != me)
            st_release_sys((uint32_t*)((char*)c.base[p] + flags_off) + ring * n + me, seq);
      }
    }
    const uint32_t* my_flags = (const uint32_t*)((const char*)c.base[me] + flags_off) + ring * n;
    if ((int)threadIdx.x < n && (int)threadIdx.x != me) spin_until(my_flags + threadIdx.x, seq, c.spin_timeout_ns);
    __syncthreads();
  }
  const char* slots = (const char*)c.base[me] + ring_off + (uint64_t)ring * n * slot_bytes;
  for (uint64_t i = i0; i < nvec; i += stride) {
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    for (int s = 0; s < n; ++s) {
      if (!(contrib >> s & 1)) continue;
      // slots written by peers during this kernel: plain (coherent) loads, not the non-coherent path
      const int4 r = (s == me) ? ld_nc_v4(partial + i * 8) : ld_v4(slots + (uint64_t)s * slot_bytes + i * 16);
      float f[8];
      unpack8h(r, f);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += f[j];
    }
    if (bias != nullptr) {
      const uint32_t c0 = (uint32_t)((i * 8) % (uint64_t)C);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += __half2float(bias[(c0 + j) % (uint32_t)C]);
    }
    if (residual != nullptr) {
      float f[8];
      unpack8h(ld_nc_v4(residual + i * 8), f);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += f[j];
    }
    st_v4(out + i * 8, pack8h(acc));
  }
}

int ar_max_ctas() {
  static int v = 0;
  if (v == 0) {
    int dev = 0, sms = 0, per_sm = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, allreduce_kernel, AR_THREADS, 0) != cudaSuccess)
      return 0;
    // every CTA of a grid that waits for the peers must be resident at once (the flags are stamped by the last CTA)
    v = sms * (per_sm < 2 ? per_sm : 2);
  }
  return v;
}

}  // namespace

extern "C" int df_allreduce_fwd(df_comm_t comm, const void* partial, void* out, int64_t rows, int C, const void* bias,
                                const void* residual, uint32_t contrib_mask, int site, int nsites, uint64_t ring_off,
                                uint64_t ring_slot_bytes, uint64_t flags_off, int ticket, void* stream) {
  const uint64_t nel = (uint64_t)rows * (uint64_t)C;
  DF_REQUIRE(out != nullptr && rows > 0 && C > 0 && nel % 8 == 0, "df_allreduce_fwd: need rows*C %% 8 == 0 (rows=%lld C=%d)",
             (long long)rows, C);
  DF_REQUIRE(((uintptr_t)partial % 16) == 0 && ((uintptr_t)out % 16) == 0 && ((uintptr_t)residual % 16) == 0,
             "df_allreduce_fwd: tensors must be 16-byte aligned");
  DF_REQUIRE(comm.world >= 1 && comm.world <= DF_MAX_WORLD && comm.rank >= 0 && comm.rank < comm.world,
             "df_allreduce_fwd: bad communicator");
  DF_REQUIRE((partial != nullptr) == ((contrib_mask >> comm.rank & 1) != 0),
             "df_allreduce_fwd: contrib_mask bit of this member must be set exactly when it passes a partial");
  if (comm.world > 1) {
    DF_REQUIRE(nel * 2 <= ring_slot_bytes, "df_allreduce_fwd: %llu bytes exceed the ring slot (%llu)",
               (unsigned long long)(nel * 2), (unsigned long long)ring_slot_bytes);
    DF_REQUIRE(site >= 0 && site < nsites && comm.clock != nullptr && comm.tickets != nullptr && ring_off % 16 == 0 &&
                   ring_slot_bytes % 16 == 0 && flags_off % 4 == 0,
               "df_allreduce_fwd: bad ring arguments");
  }
  const int max_ctas = ar_max_ctas();
  DF_REQUIRE(max_ctas > 0, "df_allreduce_fwd: cannot query the device");
  const uint64_t nvec = nel / 8;
  uint64_t need = (nvec + AR_THREADS * AR_UNROLL - 1) / (AR_THREADS * AR_UNROLL);
  const int grid = (int)(need < 1 ? 1 : (need > (uint64_t)max_ctas ? max_ctas : need));
  // launched WITHOUT the programmatic-dependent-launch attribute whatever DF_PDL says: the ring reuse relies on this kernel
  // starting only after the previous all-reduce of the stream has completed
  allreduce_kernel<<<grid, AR_THREADS, 0, (cudaStream_t)stream>>>(
      comm, (const __half*)partial, (__half*)out, nvec, C, (const __half*)bias, (const __half*)residual, contrib_mask, site,
      nsites, ring_off, ring_slot_bytes, flags_off, ticket);
  DF_CHECK_LAUNCH();
  return 0;
}
