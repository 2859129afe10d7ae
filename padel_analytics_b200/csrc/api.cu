// C-ABI surface of libpadel_b200.so: error reporting, programs (op lists), one-shot conv launches.
#include <atomic>
#include <map>
#include <memory>
#include <mutex>
#include <vector>

#include "internal.h"

namespace pb {

static thread_local std::string g_error;
std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_error = buf;
}

int num_sms() {
  static int sms = 0;
  static std::once_flag once;
  std::call_once(once, [] {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
      sms = 148;
  });
  return sms;
}

int ensure_dynamic_smem(const void* func, size_t bytes) {
  static std::mutex mu;
  static std::map<std::pair<int, const void*>, size_t> configured;
  if (bytes <= 48 * 1024) return cudaSuccess;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lk(mu);
  size_t& have = configured[{dev, func}];
  if (bytes > have) {
    e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) have = bytes;
  }
  return e;
}

enum class OpKind { Conv, MaxPool2, SppfPool };

struct Op {
  OpKind kind;
  std::unique_ptr<ConvPlan> conv;
  // pool / sppf
  const void* in = nullptr;
  void* out = nullptr;
  int N = 0, H = 0, W = 0, C = 0, c_off = 0, c = 0, out_C = 0, out_coff = 0;
};

}  // namespace pb

struct pb_program {
  std::vector<pb::Op> ops;
};

using namespace pb;

extern "C" {

const char* pb_last_error(void) { return g_error.c_str(); }

int pb_version(void) { return 101; }
long long pb_launch_count(void) { return g_launches.load(); }

int pb_conv2d(const pb_conv_desc* d, void* stream) {
  ConvPlan plan;
  if (conv_plan_build(d, &plan)) return 1;
  return conv_plan_launch(&plan, static_cast<cudaStream_t>(stream));
}

int pb_conv2d_reference(const pb_conv_desc* d, void* stream) {
  return conv_reference_launch(d, static_cast<cudaStream_t>(stream));
}

pb_program* pb_program_create(void) { return new pb_program(); }
void pb_program_destroy(pb_program* p) { delete p; }

int pb_program_add_conv(pb_program* p, const pb_conv_desc* d) {
  PB_CHECK(p && d, "program_add_conv: null argument");
  Op op;
  op.kind = OpKind::Conv;
  op.conv.reset(new ConvPlan());
  if (conv_plan_build(d, op.conv.get())) return 1;
  p->ops.push_back(std::move(op));
  return 0;
}

static int add_simple(pb_program* p, OpKind k, const void* in, int N, int H, int W, int C, int c_off, int c,
                      void* out, int out_C, int out_coff) {
  PB_CHECK(p != nullptr, "program: null");
  Op op;
  op.kind = k;
  op.in = in; op.out = out; op.N = N; op.H = H; op.W = W; op.C = C; op.c_off = c_off; op.c = c;
  op.out_C = out_C; op.out_coff = out_coff;
  p->ops.push_back(std::move(op));
  return 0;
}

int pb_program_add_maxpool2(pb_program* p, const void* in, int N, int H, int W, int C, int c_off, int c, void* out,
                            int out_C, int out_coff) {
  return add_simple(p, OpKind::MaxPool2, in, N, H, W, C, c_off, c, out, out_C, out_coff);
}
int pb_program_add_sppf_pool(pb_program* p, void* buf, int N, int H, int W, int C, int c) {
  return add_simple(p, OpKind::SppfPool, buf, N, H, W, C, 0, c, buf, C, 0);
}

int pb_program_num_ops(const pb_program* p) { return p ? (int)p->ops.size() : 0; }

int pb_program_op_kernel(const pb_program* p, int i) {
  if (!p || i < 0 || i >= (int)p->ops.size()) return -1;
  const Op& op = p->ops[i];
  switch (op.kind) {
    case OpKind::Conv: return op.conv->variant == 1 ? 1 : 0;
    case OpKind::MaxPool2: return 2;
    case OpKind::SppfPool: return 4;
  }
  return -1;
}

int pb_program_run_range(pb_program* p, int first, int last, void* stream) {
  PB_CHECK(p != nullptr, "program_run: null");
  PB_CHECK(first >= 0 && last <= (int)p->ops.size() && first <= last, "program_run: bad range");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  for (int i = first; i < last; ++i) {
    const Op& op = p->ops[i];
    int rc = 0;
    switch (op.kind) {
      case OpKind::Conv: rc = conv_plan_launch(op.conv.get(), s); break;
      case OpKind::MaxPool2:
        rc = launch_maxpool2(op.in, op.N, op.H, op.W, op.C, op.c_off, op.c, op.out, op.out_C, op.out_coff, s);
        break;
      case OpKind::SppfPool: rc = launch_sppf_pool(op.out, op.N, op.H, op.W, op.C, op.c, s); break;
    }
    if (rc) return rc;
  }
  return 0;
}

int pb_program_run(pb_program* p, void* stream) {
  return pb_program_run_range(p, 0, p ? (int)p->ops.size() : 0, stream);
}

}  // extern "C"
