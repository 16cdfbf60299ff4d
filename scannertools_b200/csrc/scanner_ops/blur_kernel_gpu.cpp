// Blur op, GPU kernel -- a GPU registration for the reference's Blur op, whose only kernel is the CPU BlurKernel
// (scannertools_cpp/imgproc/blur_kernel_cpu.cpp).  BlurArgs { int32 kernel_size = 1; float sigma = 2; }
// (scannertools_imgproc.proto) arrive in config.args and are parsed in the constructor; empty or unparsable args
// fail validate(), as in the reference (:29-33).  sigma is parsed and ignored: the reference stores it and never
// reads it, so the op is a box blur (stb_blur_u8 restates the arithmetic).  kernel_size outside 1..255 fails
// validate() too: below 1 the reference indexes out of bounds, above 255 is not supported.
#include <vector>

#include "scanner/api/kernel.h"
#include "scanner/api/op.h"
#include "scanner/util/cuda.h"
#include "scanner/util/memory.h"
#include "proto_wire.h"
#include "stb_check.h"

namespace scanner {
namespace {

// protobuf wire format of BlurArgs: 1 kernel_size (varint), 2 sigma (fixed32 as a float; fixed64 tolerated)
bool parse_blur_args(const std::vector<u8>& buf, i32* kernel_size) {
  *kernel_size = 0;
  if (buf.empty()) return false;
  return parse_wire_fields(buf, [kernel_size](const WireField& f) {
    if (f.field == 1 && f.wire == 0) *kernel_size = (i32)f.varint;
  });
}

}  // namespace

class BlurKernelGPU : public BatchedKernel {
 public:
  BlurKernelGPU(const KernelConfig& config) : BatchedKernel(config), device_(config.devices[0]) {
    valid_.set_success(true);
    if (!parse_blur_args(config.args, &kernel_size_)) {
      RESULT_ERROR(&valid_, "Blur: could not parse BlurArgs");
    } else if (kernel_size_ < 1 || kernel_size_ > 255) {
      RESULT_ERROR(&valid_, "Blur (B200): kernel_size %d is outside 1..255", kernel_size_);
    }
    CU_CHECK(cudaSetDevice(device_.id));
    CU_CHECK(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
  }

  ~BlurKernelGPU() {
    cudaSetDevice(device_.id);
    cudaStreamDestroy(stream_);
  }

  void validate(Result* result) override { result->CopyFrom(valid_); }

  void execute(const BatchedElements& input_columns, BatchedElements& output_columns) override {
    auto& frame_col = input_columns[0];
    CU_CHECK(cudaSetDevice(device_.id));
    const Frame* frame = frame_col[0].as_const_frame();
    const i32 input_count = (i32)num_rows(frame_col);
    const int ch = frame->channels();
    if (frame->type != FrameType::U8 || !(ch == 1 || ch == 3 || ch == 4)) {
      // the reference reads the frame as 3-channel bytes whatever it is; an F32 frame must not be blurred as bytes
      STB_FATAL("Blur (B200): only U8 frames with 1, 3 or 4 channels are implemented");
    }
    FrameInfo info(frame->height(), frame->width(), ch, FrameType::U8);
    std::vector<Frame*> output_frames = new_frames(device_, info, input_count);
    src_.resize(input_count);
    dst_.resize(input_count);
    for (i32 i = 0; i < input_count; ++i) {
      src_[i] = frame_col[i].as_const_frame()->data;
      dst_[i] = output_frames[i]->data;
    }
    STB_CHECK(stb_blur_u8(src_.data(), input_count, frame->width(), frame->height(), ch, kernel_size_, dst_.data(),
                          stream_));
    for (i32 i = 0; i < input_count; ++i) insert_frame(output_columns[0], output_frames[i]);
    CU_CHECK(cudaStreamSynchronize(stream_));
  }

 private:
  DeviceHandle device_;
  cudaStream_t stream_;
  i32 kernel_size_ = 0;
  Result valid_;
  std::vector<const uint8_t*> src_;
  std::vector<uint8_t*> dst_;
};

#ifndef STB_SKIP_OP_DECLARATIONS
REGISTER_OP(Blur).frame_input("frame").frame_output("frame");
#endif

REGISTER_KERNEL(Blur, BlurKernelGPU).device(DeviceType::GPU).batch().num_devices(1);

// test harness hook (compat build only): run the kernel with serialized BlurArgs
#ifdef STB_COMPAT_SHIM
extern "C" __attribute__((visibility("default"))) int stb_shim_blur(const uint8_t* h_frames, int n, int w, int h, int c,
                                                                    const uint8_t* args, int args_len, uint8_t* h_out,
                                                                    int out_capacity, int device_id) {
  KernelConfig cfg;
  cfg.devices.push_back(DeviceHandle{DeviceType::GPU, device_id});
  cfg.args.assign(args, args + args_len);
  BlurKernelGPU k(cfg);
  Result r;
  k.validate(&r);
  if (!r.success()) return -4;
  DeviceHandle dev{DeviceType::GPU, device_id};
  FrameInfo info(h, w, c, FrameType::U8);
  std::vector<Frame*> in = new_frames(dev, info, n);
  BatchedElements input(1), output(1);
  for (int i = 0; i < n; ++i) {
    CU_CHECK(cudaMemcpy(in[i]->data, h_frames + (size_t)i * info.size(), info.size(), cudaMemcpyHostToDevice));
    input[0].push_back(Element(in[i]));
  }
  k.execute(input, output);
  int rc = 0;
  if ((int)output[0].size() != n) rc = -2;
  for (int i = 0; i < n && rc == 0; ++i) {
    Frame* f = output[0][i].as_frame();
    if ((size_t)(i + 1) * f->size() > (size_t)out_capacity) { rc = -3; break; }
    CU_CHECK(cudaMemcpy(h_out + (size_t)i * f->size(), f->data, f->size(), cudaMemcpyDeviceToHost));
  }
  if (!output[0].empty()) delete_buffer(dev, output[0][0].as_frame()->data);
  for (auto& e : output[0]) delete e.as_frame();
  delete_buffer(dev, in[0]->data);
  for (Frame* f : in) delete f;
  return rc;
}
#endif  // STB_COMPAT_SHIM
}  // namespace scanner
