// Host restatement of the entry points of seganygaussians_b200/csrc/cp_async.cuh for the CPU execution shim.
// TEST INFRASTRUCTURE ONLY.  Asynchronous copies are made to land as LATE as the programming model allows: cp.async pieces
// wait in a per-thread list until that thread's cp.async.wait_group / wait_all retires their group (or the thread leaves the
// kernel).  A consumer that reads staged data before the matching wait therefore reads stale bytes.
// -DSAGARS_EMU_ASYNC_EAGER flips to the other extreme: every copy lands the moment it is issued.  A kernel that refills a buffer
// its threads are still reading -- a write-after-read hazard the "late" mode cannot see -- then computes on the wrong data.  The
// suites run the staged kernels under both extremes.
#pragma once
#include <cstring>
#include <deque>
#include <vector>

namespace sagars {

// "shared-window address" of a pointer into the block's dynamic shared memory: its offset in that buffer (what the matrix
// descriptors of tc.cuh pack; the buffer is 1024-byte aligned, so 16-byte granules line up)
inline uint32_t smem_u32(const void* p)
{
    return (uint32_t)(reinterpret_cast<uintptr_t>(p) - reinterpret_cast<uintptr_t>(::cuda_emu::dynamic_smem));
}

namespace emu_async {

struct Piece { void* dst; const void* src; int bytes = 16; };
inline thread_local std::deque<std::vector<Piece>> groups;      // committed cp.async groups, oldest first
inline thread_local std::vector<Piece> open_group;              // pieces issued since the last commit

inline void retire(std::vector<Piece>& g)
{
    for (auto& p : g) std::memcpy(p.dst, p.src, (size_t)p.bytes);
    g.clear();
}
inline void retire_all_but(size_t keep)
{
    while (groups.size() > keep) { retire(groups.front()); groups.pop_front(); }
}
inline void flush_thread()
{
    retire_all_but(0);
    retire(open_group);
}

}  // namespace emu_async

#if defined(SAGARS_EMU_ASYNC_EAGER)
inline void cp_async16(void* smem_dst, const void* gmem_src) { std::memcpy(smem_dst, gmem_src, 16); }
inline void cp_async4(void* smem_dst, const void* gmem_src) { std::memcpy(smem_dst, gmem_src, 4); }
#else
inline void cp_async16(void* smem_dst, const void* gmem_src) { emu_async::open_group.push_back({smem_dst, gmem_src}); }
inline void cp_async4(void* smem_dst, const void* gmem_src) { emu_async::open_group.push_back({smem_dst, gmem_src, 4}); }
#endif
inline void cp_async_commit()
{
    emu_async::groups.push_back(std::move(emu_async::open_group));
    emu_async::open_group.clear();
}
inline void cp_async_wait_all() { emu_async::flush_thread(); }
template <int N> inline void cp_async_wait_group() { emu_async::retire_all_but((size_t)N); }

inline void red_add(float* addr, float a)
{
    uint32_t* p = reinterpret_cast<uint32_t*>(addr);
    uint32_t old = __atomic_load_n(p, __ATOMIC_RELAXED), want;
    do {
        float f;
        std::memcpy(&f, &old, 4);
        f += a;
        std::memcpy(&want, &f, 4);
    } while (!__atomic_compare_exchange_n(p, &old, want, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED));
}
inline void red_add_v2(float* addr, float a, float b) { red_add(addr, a); red_add(addr + 1, b); }
inline void red_add_v4(float* addr, float a, float b, float c, float d) { red_add_v2(addr, a, b); red_add_v2(addr + 2, c, d); }

}  // namespace sagars
