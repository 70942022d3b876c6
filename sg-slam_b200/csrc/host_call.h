// host_call.h -- device staging of the single-call host-pointer entry points (the variants that "take HOST pointers and synchronise before
// return", include/sgs_abi.h).  A call declares each device array it needs as a slice, with its host pointer and direction; the slices share
// one cudaMalloc, freed by the destructor on every path.  Every slice starts on a 256-byte boundary -- the alignment separate cudaMallocs
// give, which the kernels' uint4 and double loads rely on -- and a slice of zero elements still gets an address of its own.
// Everything runs on the legacy default stream: upload() copies the "in" and "in-out" slices and zero-fills the slices that ask for it,
// download() copies back the "out" and "in-out" slices that have a host pointer (an "out" slice without one is device-only scratch); that
// synchronous device-to-host copy is what makes the results visible on the host.
#pragma once
#include <cuda_runtime.h>

#include <vector>

#include "sgs_common.h"

namespace sgs {

class HostCall {
  public:
    explicit HostCall(const char* fn) : fn_(fn) {}
    ~HostCall() { if (base_) cudaFree(base_); }
    HostCall(const HostCall&) = delete;
    HostCall& operator=(const HostCall&) = delete;

    // *dev receives the slice's device address in upload(); count is in elements of T
    template <class T> void in(T** dev, const void* host, size_t count) { add(dev, const_cast<void*>(host), count * sizeof(T), true, false, false); }
    template <class T> void out(T** dev, void* host, size_t count, bool zero = false) { add(dev, host, count * sizeof(T), false, true, zero); }
    template <class T> void inout(T** dev, void* host, size_t count) { add(dev, host, count * sizeof(T), true, true, false); }

    // allocates, hands out the device addresses, copies the inputs
    int upload() {
        size_t total = 0;
        for (Slice& s : s_) { s.off = total; total += ((s.bytes ? s.bytes : 1) + 255) & ~(size_t)255; }
        cudaError_t e = cudaMalloc(&base_, total);
        for (size_t i = 0; i < s_.size() && e == cudaSuccess; ++i) {
            const Slice& s = s_[i];
            s.set(s.dev, base_ + s.off);
            if (s.up && s.bytes) e = cudaMemcpy(base_ + s.off, s.host, s.bytes, cudaMemcpyHostToDevice);
            else if (s.zero) e = cudaMemset(base_ + s.off, 0, s.bytes);
        }
        return status(e);
    }

    int download() {
        cudaError_t e = cudaSuccess;
        for (size_t i = 0; i < s_.size() && e == cudaSuccess; ++i) {
            const Slice& s = s_[i];
            if (s.down && s.host && s.bytes) e = cudaMemcpy(s.host, base_ + s.off, s.bytes, cudaMemcpyDeviceToHost);
        }
        return status(e);
    }

  private:
    struct Slice {
        void* dev;
        void (*set)(void* dev, void* p);
        void* host;
        size_t bytes, off;
        bool up, down, zero;
    };
    template <class T> static void set_ptr(void* dev, void* p) { *static_cast<T**>(dev) = static_cast<T*>(p); }
    template <class T> void add(T** dev, void* host, size_t bytes, bool up, bool down, bool zero) {
        s_.push_back(Slice{dev, &set_ptr<T>, host, bytes, 0, up, down, zero});
    }
    int status(cudaError_t e) const {
        if (e == cudaSuccess) return SGS_OK;
        set_error("%s: %s", fn_, cudaGetErrorString(e));
        return SGS_ERR_CUDA;
    }

    const char* fn_;
    std::vector<Slice> s_;
    char* base_ = nullptr;
};

}  // namespace sgs
