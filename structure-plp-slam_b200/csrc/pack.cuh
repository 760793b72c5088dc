// pack.cuh -- lay many small arrays out in ONE device buffer and bind each array's device pointer where it is laid out
// (the reference-facing entry points take host pointers; per-array cudaMemcpy calls would be launch-latency bound at
// these sizes).
//
// A slot is registered with the pointer it binds, e.g. lay.in(J.qx, q->reproj_x, m) or lay.out(J.matched_out, n);
// counts are in elements of the pointer's type.  Two ways to place the layout:
//   upload(ctx, slot)  staged: sizes the context scratch slot, binds every slot, copies the inputs into the pinned
//                      buffer and issues one H2D copy.  Host tables that hold slots (job structs) are inputs too:
//                      their pointers are filled before they are copied.
//   bind(base)         a block of bytes() the caller allocated (and fills) itself.
// The addresses handed to in / out / alias must not move before the layout is placed: size job vectors first.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace plp {

class Layout {
  public:
    // n elements copied from src by upload(); a null src or n == 0 binds nullptr and takes no space
    template <typename D, typename T>
    void in(D *&dst, const T *src, size_t n) {
        static_assert(std::is_same<typename std::remove_const<D>::type, T>::value, "slot and source types differ");
        dst = nullptr;
        if (src && n) add(&dst, src, n * sizeof(T));
    }
    // output / scratch space of n elements, NOT cleared (it holds whatever the buffer held; every kernel writes its
    // outputs before anything reads them)
    template <typename T>
    void out(T *&dst, size_t n) {
        add(&dst, nullptr, n * sizeof(T));
    }
    // dst is bound to whatever `to` is bound to (one array read through two tables)
    template <typename D, typename T>
    void alias(D *&dst, T *const &to) {
        static_assert(std::is_same<typename std::remove_const<D>::type, typename std::remove_const<T>::type>::value,
                      "alias types differ");
        aliases_.push_back({(void *)&dst, (const void *)&to});
    }

    size_t bytes() const { return total_; }

    void bind(void *base) const {
        for (const Slot &s : slots_) {
            void *p = (uint8_t *)base + s.off;
            memcpy(s.dst, &p, sizeof(p));
        }
        for (const Alias &a : aliases_) memcpy(a.dst, a.to, sizeof(void *));
    }

    plp_status upload(plp_ctx *ctx, int scratch_slot) {
        void *d = nullptr, *h = nullptr;
        const size_t want = total_ ? total_ : 256;
        PLP_TRY(ctx_scratch(ctx, scratch_slot, want, &d));
        PLP_TRY(ctx_pinned(ctx, want, &h));
        bind(d);
        size_t hi = 0;
        for (const Slot &s : slots_) {
            if (!s.src) continue;
            memcpy((uint8_t *)h + s.off, s.src, s.bytes);
            if (s.off + s.bytes > hi) hi = s.off + s.bytes;
        }
        if (hi) PLP_CUDA_TRY(cudaMemcpyAsync(d, h, hi, cudaMemcpyHostToDevice, ctx->stream));
        dev_ = (uint8_t *)d;
        host_ = (uint8_t *)h;
        return PLP_OK;
    }

    // where a bound device address sits in the pinned staging buffer of the last upload() (for a batched readback)
    template <typename T>
    T *staged(T *dev_ptr) const {
        return (T *)(host_ + ((const uint8_t *)dev_ptr - dev_));
    }

  private:
    struct Slot {
        void *dst;  // the pointer to bind
        const void *src;
        size_t bytes, off;
    };
    struct Alias {
        void *dst;
        const void *to;
    };
    void add(void *dst, const void *src, size_t bytes) {
        slots_.push_back({dst, src, bytes, total_});
        total_ += (bytes + 255) & ~(size_t)255;
    }
    std::vector<Slot> slots_;
    std::vector<Alias> aliases_;
    size_t total_ = 0;
    uint8_t *dev_ = nullptr, *host_ = nullptr;
};

}  // namespace plp
