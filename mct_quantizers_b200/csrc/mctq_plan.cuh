// mctq_plan.cuh -- the host-side compiler of the grouped multi-tensor launch plans (mctq_unpack_plan in mctq_unpack.cu,
// mctq_lut_multi_plan in mctq_lutp.cu).
//
// A plan is a host blob: a 64-byte PlanHeader, then one PlanChunk per launch.  A chunk is the launch's __grid_constant__
// parameter block: its kernel variant, the tile count of every tensor and up to 64 argument blocks.  The grid is 2-D
// (y = tensor, x = tile; CTAs past a tensor's last tile exit at once).  Plan::compile implements the grouping rule that
// include/mctq.h states for both plans.
// What stays with each kind: describing one tensor (validation, variant, argument block, tiles, shared memory), mapping the
// variant to a kernel instantiation, and declaring the launch for dependent launch.
#pragma once
#include <algorithm>
#include <array>
#include <vector>

#include "mctq_common.cuh"

namespace mctq {

constexpr int kPlanMaxDesc = 64;

// Variant: seven int32, the fields that select the kernel instantiation in the order plans sort by, zero-padded
template <class Variant, class Entry, int CAP>
struct PlanChunk {
    int32_t n_desc;
    Variant var;
    int32_t tiles[CAP + 4];      // tiles[k] = tiles of tensor k; tiles[CAP] = the largest of them (grid x)
    alignas(16) Entry e[CAP];    // LUT blocks (144 bytes) stay 16-byte aligned: with 8 nvcc compiles their kernels differently
};

struct PlanHeader {          // 64 bytes
    uint32_t magic;
    int32_t n_desc, n_chunks;
    int32_t tiles_per_cta;   // LUT blobs: 1, which their readers check; unpack blobs: 0 (not recorded)
    int64_t total_tiles;
    uint64_t smem_bytes;     // the largest dynamic shared memory of any tensor's kernel
    int32_t reserved[8];
};
static_assert(sizeof(PlanHeader) == 64, "plan header layout");

template <class Variant, class Entry, uint32_t MAGIC>
struct Plan {
    using Chunk = PlanChunk<Variant, Entry, kPlanMaxDesc>;
    static_assert(sizeof(Variant) == 7 * sizeof(int32_t), "variant layout");
    static_assert(sizeof(Chunk) <= 32764, "kernel parameter space");

    // one tensor as its kind describes it; skip = nothing to launch
    struct Item {
        Entry args;
        Variant var;
        int64_t tiles;
        size_t smem;
        bool skip;
    };

    PlanHeader h = {};
    std::vector<Chunk> chunks;

    static std::array<int32_t, 7> fields(const Variant& v) {
        std::array<int32_t, 7> f;
        memcpy(f.data(), &v, sizeof(f));
        return f;
    }

    // describe(descs[k], item) -> 0 or MCTQ_E_*, called for every tensor in order before any tile count is checked
    template <class Desc, class Describe>
    int compile(const Desc* descs, int n_desc, Describe&& describe) {
        if (!descs || n_desc < 1) return MCTQ_E_BADARG;
        std::vector<Item> items((size_t)n_desc);                 // zero-filled
        std::vector<int> order;
        for (int k = 0; k < n_desc; ++k) {
            if (const int rc = describe(descs[k], items[k])) return rc;
            if (!items[k].skip) order.push_back(k);
        }
        for (const int k : order) {
            if (items[k].tiles > 0x7fffffffLL) return MCTQ_E_BADARG;
            h.smem_bytes = std::max<uint64_t>(h.smem_bytes, items[k].smem);
        }
        std::sort(order.begin(), order.end(), [&](int a, int b) {
            const auto fa = fields(items[a].var), fb = fields(items[b].var);
            if (fa != fb) return fa < fb;
            return items[a].tiles != items[b].tiles ? items[a].tiles > items[b].tiles : a < b;
        });
        for (const int k : order) {
            const Item& it = items[k];
            if (chunks.empty() || chunks.back().n_desc == kPlanMaxDesc || fields(chunks.back().var) != fields(it.var) ||
                it.tiles * 16 < chunks.back().tiles[kPlanMaxDesc]) {
                Chunk& c = chunks.emplace_back();                  // zero-filled
                c.var = it.var;
                c.tiles[kPlanMaxDesc] = (int32_t)it.tiles;
            }
            Chunk& c = chunks.back();
            c.e[c.n_desc] = it.args;
            c.tiles[c.n_desc++] = (int32_t)it.tiles;
            h.total_tiles += it.tiles;
        }
        h.magic = MAGIC;
        h.n_desc = n_desc;
        h.n_chunks = (int32_t)chunks.size();
        return 0;
    }

    size_t bytes() const { return sizeof(PlanHeader) + chunks.size() * sizeof(Chunk); }

    // the blob into the caller's buffer; the total tile count or MCTQ_E_BADARG
    int64_t write(void* out, size_t out_bytes) const {
        if (!out || out_bytes < bytes()) return MCTQ_E_BADARG;
        memcpy(out, &h, sizeof(PlanHeader));
        if (!chunks.empty()) memcpy(reinterpret_cast<uint8_t*>(out) + sizeof(PlanHeader), chunks.data(), chunks.size() * sizeof(Chunk));
        return h.total_tiles;
    }

    // launch(chunk, header) for every chunk of a blob, the chunk copied into a parameter block of SMALL or 64 tensors (the
    // block is copied by every launch); 0, MCTQ_E_BADARG for a blob that is not a plan of this kind, or launch's error
    template <int SMALL, class Launch>
    static int run(const void* blob, int min_chunks, Launch&& launch) {
        if (!blob) return MCTQ_E_BADARG;
        const PlanHeader* hb = reinterpret_cast<const PlanHeader*>(blob);
        if (hb->magic != MAGIC || hb->n_desc < 1 || hb->n_chunks < min_chunks) return MCTQ_E_BADARG;
        const Chunk* cs = reinterpret_cast<const Chunk*>(reinterpret_cast<const uint8_t*>(blob) + sizeof(PlanHeader));
        for (int c = 0; c < hb->n_chunks; ++c) {
            const int rc = cs[c].n_desc <= SMALL ? launch(copy<SMALL>(cs[c]), *hb) : launch(copy<kPlanMaxDesc>(cs[c]), *hb);
            if (rc) return rc;
        }
        return 0;
    }

    template <int CAP>
    static PlanChunk<Variant, Entry, CAP>& copy(const Chunk& c) {
        static thread_local PlanChunk<Variant, Entry, CAP> p;   // up to 10 KB: not on the stack
        p.n_desc = c.n_desc;
        p.var = c.var;
        memcpy(p.tiles, c.tiles, (size_t)c.n_desc * sizeof(int32_t));
        p.tiles[CAP] = c.tiles[kPlanMaxDesc];
        memcpy(p.e, c.e, (size_t)c.n_desc * sizeof(Entry));
        return p;
    }
};

}  // namespace mctq
