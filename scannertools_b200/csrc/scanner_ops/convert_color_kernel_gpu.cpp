// ConvertColor op, GPU kernel -- drop-in for the GPU registration of the reference's
// ConvertColorKernel (scannertools_cpp/imgproc/convert_color_kernel.cpp:200-300): per-stream
// ConvertColorArgs { string conversion = 1 } (scannertools_imgproc.proto:29-31) arrive through
// new_stream(args); unknown / unimplemented conversion names are reported through validate(),
// as the reference does (:238-243).  Also registers a GPU kernel for the legacy ConvertToHSVCPP
// op (scannertools/old/cpp_ops/imgproc.cpp:14-48, 236-243: cv::cvtColor(.., COLOR_RGB2HSV)),
// which is CPU-only in the reference.
#include <memory>
#include <string>
#include <vector>

#include "scanner/api/kernel.h"
#include "scanner/api/op.h"
#include "scanner/util/cuda.h"
#include "scanner/util/memory.h"
#include "stb_check.h"

namespace scanner {
namespace {

// protobuf wire format: field 1, length-delimited string
bool parse_conversion(const std::vector<u8>& buf, std::string* out) {
  size_t p = 0;
  while (p < buf.size()) {
    const u8 key = buf[p++];
    if ((key & 7) != 2) return false;
    u64 len = 0;
    int shift = 0;
    while (p < buf.size()) {
      const u8 b = buf[p++];
      len |= (u64)(b & 0x7f) << shift;
      shift += 7;
      if (!(b & 0x80)) break;
    }
    if (len > buf.size() - p) return false;
    if ((key >> 3) == 1) out->assign(reinterpret_cast<const char*>(buf.data() + p), (size_t)len);
    p += (size_t)len;
  }
  return true;
}

}  // namespace

class ConvertColorKernelGPU : public BatchedKernel {
 public:
  ConvertColorKernelGPU(const KernelConfig& config, const char* fixed_conversion = nullptr)
    : BatchedKernel(config), device_(config.devices[0]), code_(-1) {
    valid_.set_success(true);
    CU_CHECK(cudaSetDevice(device_.id));
    CU_CHECK(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
    if (fixed_conversion) set_conversion(fixed_conversion);
  }

  ~ConvertColorKernelGPU() {
    cudaSetDevice(device_.id);
    cudaStreamDestroy(stream_);
  }

  void validate(Result* result) override { result->CopyFrom(valid_); }

  int code() const { return code_; }

  void new_stream(const std::vector<u8>& args) {
    std::string conv;
    if (!parse_conversion(args, &conv)) { RESULT_ERROR(&valid_, "ConvertColor: could not parse ConvertColorArgs"); return; }
    set_conversion(conv);
  }

  void execute(const BatchedElements& input_columns, BatchedElements& output_columns) override {
    auto& frame_col = input_columns[0];
    CU_CHECK(cudaSetDevice(device_.id));
    const Frame* frame = frame_col[0].as_const_frame();
    const i32 input_count = (i32)num_rows(frame_col);
    const int in_channels = stb_color_in_channels(code_);
    if (frame->type != FrameType::U8 || frame->channels() != in_channels) {
      // cv::cvtColor rejects a frame whose depth or channel count does not fit the conversion
      char msg[256];
      snprintf(msg, sizeof(msg), "ConvertColor (B200): %s needs %d-channel U8 frames, got %s frames with %d channels",
               conversion_.c_str(), in_channels, frame->type == FrameType::U8 ? "U8" : "non-U8", (int)frame->channels());
      STB_FATAL(msg);
    }
    FrameInfo info(frame->height(), frame->width(), stb_color_out_channels(code_), FrameType::U8);
    std::vector<Frame*> output_frames = new_frames(device_, info, input_count);
    src_.resize(input_count);
    dst_.resize(input_count);
    for (i32 i = 0; i < input_count; ++i) {
      src_[i] = frame_col[i].as_const_frame()->data;
      dst_[i] = output_frames[i]->data;
    }
    STB_CHECK(stb_convert_color_u8(src_.data(), input_count, frame->width(), frame->height(), code_, dst_.data(), stream_));
    for (i32 i = 0; i < input_count; ++i) insert_frame(output_columns[0], output_frames[i]);
    CU_CHECK(cudaStreamSynchronize(stream_));
  }

 private:
  void set_conversion(const std::string& conv) {
    conversion_ = conv;
    code_ = stb_color_code(conv.c_str());
    if (code_ < 0) RESULT_ERROR(&valid_, "ConvertColor (B200): conversion type %s is not implemented", conv.c_str());
  }

  DeviceHandle device_;
  cudaStream_t stream_;
  int code_;
  std::string conversion_;
  Result valid_;
  std::vector<const uint8_t*> src_;
  std::vector<uint8_t*> dst_;
};

class ConvertToHSVKernelGPU : public ConvertColorKernelGPU {
 public:
  ConvertToHSVKernelGPU(const KernelConfig& config) : ConvertColorKernelGPU(config, "COLOR_RGB2HSV") {}
};

#ifndef STB_SKIP_OP_DECLARATIONS
REGISTER_OP(ConvertColor).frame_input("frame").frame_output("frame");
REGISTER_OP(ConvertToHSVCPP).frame_input("frame").frame_output("frame");
#endif

REGISTER_KERNEL(ConvertColor, ConvertColorKernelGPU).device(DeviceType::GPU).batch().num_devices(1);
REGISTER_KERNEL(ConvertToHSVCPP, ConvertToHSVKernelGPU).device(DeviceType::GPU).batch().num_devices(1);

// test harness hook (compat build only)
#ifdef STB_COMPAT_SHIM
extern "C" __attribute__((visibility("default"))) int stb_shim_convert_color(const uint8_t* h_frames, int n, int w, int h,
                                                                             const uint8_t* args, int args_len,
                                                                             uint8_t* h_out, int* out_channels, int device_id) {
  KernelConfig cfg;
  cfg.devices.push_back(DeviceHandle{DeviceType::GPU, device_id});
  std::unique_ptr<ConvertColorKernelGPU> k;
  if (args_len < 0) k.reset(new ConvertToHSVKernelGPU(cfg));
  else { k.reset(new ConvertColorKernelGPU(cfg)); k->new_stream(std::vector<u8>(args, args + args_len)); }
  Result r;
  k->validate(&r);
  if (!r.success()) return -4;
  DeviceHandle dev{DeviceType::GPU, device_id};
  FrameInfo info(h, w, stb_color_in_channels(k->code()), FrameType::U8);
  std::vector<Frame*> in = new_frames(dev, info, n);
  BatchedElements input(1), output(1);
  for (int i = 0; i < n; ++i) {
    CU_CHECK(cudaMemcpy(in[i]->data, h_frames + (size_t)i * info.size(), info.size(), cudaMemcpyHostToDevice));
    input[0].push_back(Element(in[i]));
  }
  k->execute(input, output);
  int rc = (int)output[0].size() == n ? 0 : -2;
  for (int i = 0; i < n && rc == 0; ++i) {
    Frame* f = output[0][i].as_frame();
    *out_channels = f->channels();
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
