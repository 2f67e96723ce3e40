// tcgen05 attention core (head size 32 with an even head count, or 64; T in {16,32,64,128,256}) on the internal NHWC bf16 qkv tensor; see attn_tc.cu.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

namespace ub {

struct AttnTcParams {
    CUtensorMap tmQKV;  // qkv  [B*T][3C] bf16, box (64 channels, 128 rows), SWIZZLE_128B
    CUtensorMap tmDO;   // dout [B*T][C]  bf16, same box (backward only)
    const __nv_bfloat16* qkv;
    int ld;
    int B, T, NH, tshift;
    __nv_bfloat16* out;  // [B*T][ldo]  attention output (written by forward, read by backward)
    int ldo;
    float* lse;          // [B][NH][T] log2-domain logsumexp of the scaled scores
    const __nv_bfloat16* dout;
    int lddo;
    __nv_bfloat16* dqkv;  // [B*T][ldd], sections [dQ | dK | dV]
    int ldd;
    float* dsum;          // [B][NH][T] rowsum(dO o O), written by the dq kernel (the dkv kernel recomputes it)
    int HS;               // head size, 32 or 64 (selects the kernel instantiation)
};

bool attn_tc_supported(int T, int NH, int HS);
void attn_tc_init();
// dout / dqkv / dsum may be null for a forward-only plan.
int attn_tc_plan(AttnTcParams* p, const __nv_bfloat16* qkv, int ld, int B, int T, int NH, int HS, __nv_bfloat16* out,
                 int ldo, float* lse, const __nv_bfloat16* dout, int lddo, __nv_bfloat16* dqkv, int ldd, float* dsum);
int attn_tc_fwd(const AttnTcParams& p, cudaStream_t st);
int attn_tc_bwd(const AttnTcParams& p, cudaStream_t st, cudaStream_t aux = nullptr, cudaEvent_t ev_fork = nullptr,
                cudaEvent_t ev_join = nullptr);

}  // namespace ub
