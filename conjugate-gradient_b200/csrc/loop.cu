// loop.cu -- the small kernels of a device solve (cgb_solve_device, cgb_solve_block_device): the
// host neither polls a flag nor counts loop bodies, so the loop's bookkeeping lives on the device.
//   device_begin  the State(s) a solve starts from and the loop's body limit, from kernel arguments
//   loop_ctl      bodies run so far, and the condition of a CUDA-graph WHILE node: go on while the
//                 stop test has not fired and a whole body still fits under max_iter
//   device_info   cgb_solve_info and the r'r history of every column into the caller's device memory
#include "../../include/cgb200.h"
#include "cgb_kernels.h"

namespace cgb {

namespace {

__global__ void __launch_bounds__(32) device_begin_kernel(State *st, int nst, LoopCtl *ctl, long long max_iter)
{
    const int j = threadIdx.x;
    if (j < nst) { // what cgb_solve_begin / cgb_solve_block_begin upload
        State s;
        s.rsold = s.rsnew = s.conj = s.alpha = 0.0;
        s.iter = -1;
        s.done = 0;
        s.pad = 0;
        st[j] = s;
    }
    if (j == 0) {
        ctl->limit = max_iter;
        ctl->bodies = 0;
        ctl->t0 = 0;
    }
}

__global__ void __launch_bounds__(32) loop_ctl_kernel(LoopCtl *ctl, const int *done, const unsigned int *ndone, int nrhs,
                                                      cudaGraphConditionalHandle h, int set, int len, int add, int reset)
{
    if (threadIdx.x != 0) return;
    const long long n = reset ? 0 : ctl->bodies + add;
    ctl->bodies = n;
    if (reset) ctl->t0 = globaltimer_ns();
    if (!set) return;
    // the kernels before this one have completed: `done` / the count of converged columns is final
    const bool fin = done ? *(volatile const int *)done != 0 : *(volatile const unsigned int *)ndone >= (unsigned)nrhs;
    cudaGraphSetConditional(h, (!fin && ctl->limit - n >= len) ? 1u : 0u);
}

// one block: warp j reports column j
__global__ void __launch_bounds__(kMaxRhs * 32) device_info_kernel(const State *st, int nrhs, const LoopCtl *ctl,
                                                                   cgb_solve_info *info, const double *hist,
                                                                   long long hist_ld, double *hist_out, long long out_ld)
{
    __shared__ unsigned long long t1;
    if (threadIdx.x == 0) t1 = globaltimer_ns();
    __syncthreads();
    const int j = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (j >= nrhs) return;
    const State s = st[j];
    const long long executed = s.done ? s.iter + 1 : s.iter; // as cgb_solve_end
    if (lane == 0) {
        cgb_solve_info o;
        o.k = s.iter;
        o.converged = s.done;
        o.rsold = s.rsold;
        o.rsnew = s.rsnew;
        o.seconds = ctl->t0 ? (double)(t1 - ctl->t0) * 1e-9 : 0.0;
        o.iterations = executed;
        info[j] = o;
    }
    if (hist && hist_out)
        for (long long t = lane; t < executed; t += 32) hist_out[j * out_ld + t] = hist[j * hist_ld + t];
}

} // namespace

cudaError_t preload_loop_kernels()
{
    cudaFuncAttributes fa;
    cudaError_t e;
    if ((e = cudaFuncGetAttributes(&fa, device_begin_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&fa, loop_ctl_kernel)) != cudaSuccess) return e;
    return cudaFuncGetAttributes(&fa, device_info_kernel);
}

cudaError_t launch_device_begin(State *st, int nst, LoopCtl *ctl, long long max_iter, cudaStream_t s)
{
    device_begin_kernel<<<1, 32, 0, s>>>(st, nst, ctl, max_iter);
    return cudaGetLastError();
}

cudaError_t launch_loop_ctl(LoopCtl *ctl, const int *done, const unsigned int *ndone, int nrhs,
                            cudaGraphConditionalHandle h, int set, int len, int add, int reset, cudaStream_t s)
{
    loop_ctl_kernel<<<1, 32, 0, s>>>(ctl, done, ndone, nrhs, h, set, len, add, reset);
    return cudaGetLastError();
}

cudaError_t launch_device_info(const State *st, int nrhs, const LoopCtl *ctl, cgb_solve_info *info, const double *hist,
                               long long hist_ld, double *hist_out, long long out_ld, cudaStream_t s)
{
    device_info_kernel<<<1, kMaxRhs * 32, 0, s>>>(st, nrhs, ctl, info, hist, hist_ld, hist_out, out_ld);
    return cudaGetLastError();
}

} // namespace cgb
