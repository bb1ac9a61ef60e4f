// Export / import of per-stream carried state: one table-driven gather (pack) and scatter (unpack) for the CRN and
// FullSubNet contexts (se_crn_state_export / _import, se_fsn_state_export / _import).
//
// A context describes its carried state as a StateTable (se_internal.h): one entry per buffer, giving where the bytes
// of row r sit.  A record is the entries of one row packed back to back in table order, each padded to 16 bytes, so
// its layout depends on the table alone, not on max_streams or the device: export -> import -> export gives identical
// bytes, and a record moves between contexts of different capacity and between GPUs.
//
// grid (slices, rows): a block moves one 16 KB slice of one entry of one row; the launcher lays the entries' slices end
// to end (no empty blocks).  Each thread has 64 bytes in flight (four 16-byte or sixteen 4-byte loads) before its
// first store.  The row list travels by value in the kernel parameters (up to kRowsPerLaunch rows per launch, within
// the 32 KB parameter limit of CUDA 12.1+), so nothing is staged in a buffer that a later call could overwrite.
#include <cuda_runtime.h>
#include <string.h>

#include <string>
#include <type_traits>
#include <vector>

#include "se_internal.h"

namespace se {

namespace {

constexpr int kSliceBytes = 16384;
constexpr int kThreads = 256;
constexpr int kRowsPerLaunch = 7168;

struct StateArgs {
    StateEntry e[kMaxStateEntries];
    int first_block[kMaxStateEntries + 1];
    int n_entries, record_bytes;
    char* rec;
    int rows[kRowsPerLaunch];
};
static_assert(sizeof(StateArgs) <= 32764, "kernel parameters are limited to 32764 bytes");

template <typename V, bool kPack>
__device__ __forceinline__ void copy_slice(const StateEntry& e, char* row, char* rec, int j0) {
    constexpr int kPer = 64 / (int)sizeof(V);
    const int bytes = e.run * e.count;
    const int seg = (bytes + 15) & ~15;
    V v[kPer];
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
        const int j = j0 + (int)sizeof(V) * (threadIdx.x + kThreads * k);
        v[k] = V();
        if (j < bytes) {
            const int u = j / e.run;
            char* arena = row + (long long)u * e.unit_stride + (j - u * e.run);
            v[k] = kPack ? *reinterpret_cast<const V*>(arena) : *reinterpret_cast<const V*>(rec + j);
        }
    }
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
        const int j = j0 + (int)sizeof(V) * (threadIdx.x + kThreads * k);
        if (kPack) {
            if (j < seg) *reinterpret_cast<V*>(rec + j) = v[k];  // the padding of the segment is written as zeros
        } else if (j < bytes) {
            const int u = j / e.run;
            *reinterpret_cast<V*>(row + (long long)u * e.unit_stride + (j - u * e.run)) = v[k];
        }
    }
}

template <bool kPack>
__global__ void __launch_bounds__(kThreads) state_copy_kernel(const __grid_constant__ StateArgs a) {
    int ei = 0;
    while (ei + 1 < a.n_entries && (int)blockIdx.x >= a.first_block[ei + 1]) ++ei;
    const StateEntry& e = a.e[ei];
    const int i = blockIdx.y;
    char* row = e.base + (long long)a.rows[i] * e.row_stride;
    char* rec = a.rec + (long long)i * a.record_bytes + e.rec_off;
    const int j0 = ((int)blockIdx.x - a.first_block[ei]) * kSliceBytes;
    if (e.vec == 16) copy_slice<uint4, kPack>(e, row, rec, j0);
    else copy_slice<uint32_t, kPack>(e, row, rec, j0);
}

int launch_state_copy(const StateTable& t, const int32_t* rows, int n, char* rec, bool pack, cudaStream_t st) {
    if (n == 0 || t.n == 0) return 0;
    static_assert(std::is_trivially_copyable<StateArgs>::value, "kernel parameter");
    std::vector<char> storage(sizeof(StateArgs));  // 32 KB: kept off the host stack
    StateArgs& a = *reinterpret_cast<StateArgs*>(storage.data());
    int blocks = 0;
    for (int i = 0; i < t.n; ++i) {
        a.e[i] = t.e[i];
        a.first_block[i] = blocks;
        blocks += ((t.e[i].run * t.e[i].count + 15) / 16 * 16 + kSliceBytes - 1) / kSliceBytes;
    }
    a.first_block[t.n] = blocks;
    a.n_entries = t.n;
    a.record_bytes = t.record_bytes;
    for (int off = 0; off < n; off += kRowsPerLaunch) {
        const int nb = (n - off) < kRowsPerLaunch ? (n - off) : kRowsPerLaunch;
        memcpy(a.rows, rows + off, (size_t)nb * sizeof(int32_t));
        a.rec = rec + (long long)off * t.record_bytes;
        if (pack) state_copy_kernel<true><<<dim3(blocks, nb), kThreads, 0, st>>>(a);
        else state_copy_kernel<false><<<dim3(blocks, nb), kThreads, 0, st>>>(a);
        SE_CUDA_OK(cudaGetLastError());
    }
    return 0;
}

}  // namespace

int state_table_add(StateTable& t, const std::string& name, int esz, void* base, long long row_stride, long long run,
                    int count, long long unit_stride) {
    SE_REQUIRE(t.n < kMaxStateEntries, "internal: state table full");
    SE_REQUIRE(base != nullptr && run > 0 && count > 0 && run * count < (1LL << 30), "internal: state entry " + name);
    SE_REQUIRE(reinterpret_cast<uintptr_t>(base) % 4 == 0 && row_stride % 4 == 0 && unit_stride % 4 == 0 && run % 4 == 0,
               "internal: state entry " + name + " is not 4-byte aligned");
    StateEntry& e = t.e[t.n++];
    e.base = static_cast<char*>(base);
    e.row_stride = row_stride;
    e.unit_stride = count > 1 ? unit_stride : 0;
    e.run = (int)run;
    e.count = count;
    e.rec_off = t.record_bytes;
    const bool v16 = reinterpret_cast<uintptr_t>(base) % 16 == 0 && row_stride % 16 == 0 && e.unit_stride % 16 == 0 &&
                     run % 16 == 0;
    e.vec = v16 ? 16 : 4;
    t.record_bytes += (int)((run * count + 15) / 16 * 16);
    t.desc += " " + name + ":" + std::to_string(esz) + ":" + std::to_string(count) + "x" + std::to_string(run) + "@" +
              std::to_string(e.rec_off);
    return 0;
}

uint64_t state_layout_hash(const StateTable& t) {
    uint64_t h = 1469598103934665603ull;
    for (unsigned char ch : t.desc) {
        h ^= ch;
        h *= 1099511628211ull;
    }
    return h;
}

int state_rows_check(const int32_t* rows, int n, int max_streams, bool unique, const char* what) {
    SE_REQUIRE(n >= 0, std::string(what) + ": negative row count");
    SE_REQUIRE(n == 0 || rows != nullptr, std::string(what) + ": null row list");
    std::vector<char> seen(unique ? max_streams : 0, 0);
    for (int i = 0; i < n; ++i) {
        SE_REQUIRE(rows[i] >= 0 && rows[i] < max_streams, std::string(what) + ": row " + std::to_string(rows[i]) +
                                                              " outside [0, " + std::to_string(max_streams) + ")");
        if (unique) {
            SE_REQUIRE(!seen[rows[i]], std::string(what) + ": row " + std::to_string(rows[i]) + " appears twice");
            seen[rows[i]] = 1;
        }
    }
    return 0;
}

int launch_state_pack(const StateTable& t, const int32_t* rows, int n, void* rec, cudaStream_t st) {
    return launch_state_copy(t, rows, n, static_cast<char*>(rec), true, st);
}
int launch_state_unpack(const StateTable& t, const int32_t* rows, int n, const void* rec, cudaStream_t st) {
    return launch_state_copy(t, rows, n, const_cast<char*>(static_cast<const char*>(rec)), false, st);
}

}  // namespace se
