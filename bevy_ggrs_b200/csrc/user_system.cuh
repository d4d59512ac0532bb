// Device API of user-defined GgrsSchedule systems (bgr_add_user_system, include/bevy_ggrs_b200.h).
//
// A user system is CUDA source registered at run time.  bgr_build puts this header, every user source (each in its own
// namespace, behind a `#line 1 "NAME"`) and one dispatcher per system into the prelude of the registration's own kernel
// (generic_program_jit.cuh), so the system runs on the register copy of a row exactly like the compiled-in systems:
//
//     BGR_SYSTEM_FN void apply_drag(const bgr_sys_ctx& ctx, bgr_commands& cmd, Velocity& v, const Ttl& t);
//
// One parameter per bound column, in binding order: `T&` is `&mut T`, `const T&` is `&T` (never written back).
// The header also parses as plain C++17 (g++), where BGR_SYSTEM_FN is `inline`: the same source then runs on the CPU.
#pragma once
#if defined(__CUDACC_RTC__)
#include "rtc_prelude.cuh"
#else
#include <cstdint>
#include <cstring>
#endif

#if defined(__CUDACC__) || defined(__CUDACC_RTC__)
#define BGR_SYSTEM_FN __device__ __forceinline__
#define BGR_SYS_HD __host__ __device__ __forceinline__
#else
#define BGR_SYSTEM_FN inline
#define BGR_SYS_HD inline
#endif

// What one system sees of the frame and of its entity.
struct bgr_sys_ctx {
    float dt;              // Time<GgrsTime>::delta_secs of this frame
    int32_t frame;         // RollbackFrameCount inside AdvanceWorld (after the frame's `+= 1`)
    uint32_t n_players;    // PlayerInputs<T>.len()
    uint8_t inputs[8];     // PlayerInputs<T>.0[handle].0
    uint64_t order;        // RollbackOrdered index of the entity (order_base + row): the player handle in box_game
    uint32_t params[8];    // the registration's parameters (compile-time constants in the generated kernel)
};

// Commands of one entity.  despawn() is deferred to after the last system of the frame.
struct bgr_commands {
    bool despawn_requested;
    BGR_SYS_HD void despawn() { despawn_requested = true; }
};

// A parameter's bit pattern as an f32, identical on the GPU and the CPU.
BGR_SYS_HD float bgr_f32(uint32_t bits) {
#if defined(__CUDA_ARCH__)
    return __uint_as_float(bits);
#else
    float f;
    memcpy(&f, &bits, 4);
    return f;
#endif
}

// ---- signature introspection (shared by the generated kernel and CPU hosts of the same source) ----
template <class T> struct bgr_param;  // only references bind: `T&` (written back) or `const T&` (read only)
template <class T> struct bgr_param<T&> { using type = T; static constexpr bool writes = true; };
template <class T> struct bgr_param<const T&> { using type = T; static constexpr bool writes = false; };

template <int I, class... A> struct bgr_nth;
template <class H, class... A> struct bgr_nth<0, H, A...> { using type = H; };
template <int I, class H, class... A> struct bgr_nth<I, H, A...> { using type = typename bgr_nth<I - 1, A...>::type; };

// void NAME(const bgr_sys_ctx&, bgr_commands&, A...): anything else leaves this incomplete (a compile error)
template <class F> struct bgr_fn_traits;
template <class... A> struct bgr_fn_traits<void (*)(const bgr_sys_ctx&, bgr_commands&, A...)> {
    static constexpr int arity = int(sizeof...(A));
    template <int I> using arg = typename bgr_nth<I, A...>::type;
    template <int I> using elem = typename bgr_param<arg<I>>::type;
};

// Defined by the generated prelude for every user system S: `run(words, on, ctx, kill)` on one row.
template <int S> struct bgr_user_system;

#if defined(__CUDACC_RTC__)
// ---- invocation glue of the generated kernel: the row is an array of words in registers ----
// Every plane index is a literal, so after inlining the typed locals are the row's registers again.
template <int P, class A> struct bgr_slot { typename bgr_param<A>::type v; };
template <class... S> struct bgr_slots : S... {};

template <int P, class A, int N>
__device__ __forceinline__ void bgr_slot_load(bgr_slot<P, A>& s, const uint32_t (&w)[N]) {
    memcpy(&s.v, &w[P], sizeof(s.v));
}
template <int P, class A, int N>
__device__ __forceinline__ void bgr_slot_store(const bgr_slot<P, A>& s, uint32_t (&w)[N], bool on) {
    if constexpr (bgr_param<A>::writes) {
        constexpr int W = int((sizeof(s.v) + 3) / 4);
        uint32_t t[W];
#pragma unroll
        for (int j = 0; j < W; ++j) t[j] = w[P + j];  // bytes of a last partial word stay as they were
        memcpy(t, &s.v, sizeof(s.v));
#pragma unroll
        for (int j = 0; j < W; ++j) w[P + j] = on ? t[j] : w[P + j];
    }
}

template <auto F, class Fn = decltype(F)> struct bgr_invoke;
template <auto F, class... A> struct bgr_invoke<F, void (*)(const bgr_sys_ctx&, bgr_commands&, A...)> {
    // P...: first word plane of each bound column.  The system runs on every row; its writes and its despawn command
    // only take effect where `on` (the row exists and has every bound column).
    template <int... P, int N>
    static __device__ __forceinline__ void run(uint32_t (&w)[N], bool on, const bgr_sys_ctx& ctx, bool& kill) {
        static_assert(sizeof...(P) == sizeof...(A), "one word plane per bound column");
        bgr_slots<bgr_slot<P, A>...> s;
        (bgr_slot_load(static_cast<bgr_slot<P, A>&>(s), w), ...);
        bgr_commands cmd{false};
        F(ctx, cmd, static_cast<bgr_slot<P, A>&>(s).v...);
        (bgr_slot_store(static_cast<bgr_slot<P, A>&>(s), w, on), ...);
        kill = kill || (on && cmd.despawn_requested);
    }
};
#endif
