// Process-wide C-ABI helpers.
#include "common.cuh"

extern "C" const char* koe_last_error(void) { return koe::err_buf(); }
extern "C" int koe_version(void) { return 101; }
extern "C" int64_t koe_launch_count(void) { return koe::launch_counter().load(); }
extern "C" void koe_reset_launch_count(void) { koe::launch_counter().store(0); }
extern "C" int koe_sizeof_struct(int which) {
  switch (which) {
    case 0: return (int)sizeof(koe_frontend_config);
    case 1: return (int)sizeof(koe_logmel_args);
    case 2: return (int)sizeof(koe_core_weights);
    case 3: return (int)sizeof(koe_stream_args);
    case 4: return (int)sizeof(koe_forward_args);
    case 5: return (int)sizeof(koe_stream_pool_args);
    case 6: return (int)sizeof(koe_forward_varlen_args);
    default: return -1;
  }
}
