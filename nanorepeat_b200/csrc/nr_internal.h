// nr_internal.h -- the few host-side services of nr_api.cu that the other host translation units use (context, error
// reporting, 2-bit packing, the caching allocator).  Not part of the C ABI.
#pragma once
#include "../../include/nanorepeat_b200.h"
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

namespace nri {
int ensure_init();                               // lazy CUDA initialisation; sets this thread's device
cudaStream_t stream();                           // the library's stream
int sm_count();
int fail_msg(int code, const char* msg);         // records the thread's last error, returns code
int last_code();
bool pack(const char* s, int len, uint32_t* w);  // 16 bases per word, MSB first; false: a base other than ACGT was seen
void ambiguity(const char* s, int len, uint32_t* m);   // bit plane of the bases that are not ACGT
int alloc(void** p, size_t bytes, bool pinned);
void release(void* p, size_t bytes, bool pinned);
int check(const nr_scoring_t* sc);
void set_last_stats(const nr_stats_t& st);       // what nr_last_stats reports on this thread
}  // namespace nri
