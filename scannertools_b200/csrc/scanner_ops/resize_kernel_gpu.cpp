// Resize op, GPU kernel -- drop-in for the GPU registration of the reference's ResizeKernel
// (scannertools_cpp/imgproc/resize_kernel.cpp:22-105): per-stream ResizeArgs (width, height,
// min, preserve_aspect, interpolation; scannertools_imgproc.proto:33-39) arrive through
// new_stream(args) as a serialized protobuf; target-size rules and the batched output layout
// are the reference's; cvc::resize (:75-79) is replaced by stb_resize_u8 on 8-bit frames and stb_resize_f32 on
// float frames (OpticalFlow's H x W x 2 fields).
// The five fields are decoded with the wire-format reader of proto_wire.h, so the kernel does not
// need the generated scannertools_imgproc.pb.h.
#include <cstdio>
#include <string>
#include <vector>

#include "scanner/api/kernel.h"
#include "scanner/api/op.h"
#include "scanner/util/cuda.h"
#include "scanner/util/memory.h"
#include "proto_wire.h"
#include "stb_check.h"

namespace scanner {
namespace {

struct ResizeArgsLite {
  i32 width = 0, height = 0;
  bool min = false, preserve_aspect = false;
  std::string interpolation;
};

// protobuf wire format of ResizeArgs: 1 width (varint), 2 height (varint), 3 min (varint),
// 4 preserve_aspect (varint), 5 interpolation (length-delimited)
bool parse_resize_args(const std::vector<u8>& buf, ResizeArgsLite* out) {
  return parse_wire_fields(buf, [out](const WireField& f) {
    if (f.wire == 0) {
      if (f.field == 1) out->width = (i32)f.varint;
      else if (f.field == 2) out->height = (i32)f.varint;
      else if (f.field == 3) out->min = f.varint != 0;
      else if (f.field == 4) out->preserve_aspect = f.varint != 0;
    } else if (f.wire == 2 && f.field == 5) {
      out->interpolation.assign(reinterpret_cast<const char*>(f.data), f.len);
    }
  });
}

const char* frame_type_name(FrameType t) {
  return t == FrameType::U8 ? "U8" : t == FrameType::F32 ? "F32" : t == FrameType::F64 ? "F64" : "unknown";
}

}  // namespace

class ResizeKernelGPU : public BatchedKernel {
 public:
  ResizeKernelGPU(const KernelConfig& config) : BatchedKernel(config), device_(config.devices[0]) {
    valid_.set_success(true);
    CU_CHECK(cudaSetDevice(device_.id));
    CU_CHECK(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
  }

  ~ResizeKernelGPU() {
    cudaSetDevice(device_.id);
    cudaStreamDestroy(stream_);
  }

  void validate(Result* result) override { result->CopyFrom(valid_); }

  // Scanner calls this with the per-stream serialized ResizeArgs (resize_kernel.cpp:28-35)
  void new_stream(const std::vector<u8>& args) {
    args_ = ResizeArgsLite();
    if (!parse_resize_args(args, &args_)) RESULT_ERROR(&valid_, "Resize: could not parse ResizeArgs");
    // resize_kernel.cpp:31-35: names outside its INTERP_TYPES table silently mean INTER_LINEAR.  Of the
    // names inside the table, the five interpolation modes (INTER_NEAREST / LINEAR / CUBIC / AREA / LANCZOS4) are
    // implemented; the rest (INTER_MAX, WARP_*: flag values, not modes) fail validate() instead of silently
    // producing a different interpolation.
    interp_ = 0;
    const int code = stb_resize_interp_code(args_.interpolation.c_str());
    if (code >= 0) {
      interp_ = code;
    } else {
      static const char* const kKnownUnimplemented[] = {"INTER_MAX", "WARP_FILL_OUTLIERS", "WARP_INVERSE_MAP"};
      for (const char* name : kKnownUnimplemented)
        if (args_.interpolation == name)
          RESULT_ERROR(&valid_, "Resize (B200): interpolation %s is not implemented (INTER_NEAREST, INTER_LINEAR, INTER_CUBIC, INTER_AREA, INTER_LANCZOS4)",
                       args_.interpolation.c_str());
    }
  }

  void execute(const BatchedElements& input_columns, BatchedElements& output_columns) override {
    auto& frame_col = input_columns[0];
    CU_CHECK(cudaSetDevice(device_.id));
    const Frame* frame = frame_col[0].as_const_frame();

    i32 target_width = 0, target_height = 0;
    STB_CHECK(stb_resize_target(frame->width(), frame->height(), args_.width, args_.height, args_.min ? 1 : 0,
                                args_.preserve_aspect ? 1 : 0, &target_width, &target_height));
    const i32 input_count = (i32)num_rows(frame_col);
    const int ch = frame->channels();
    // resize_kernel.cpp:64 propagates frame->type to cv::resize: 8-bit frames with 1, 3 or 4 channels and float
    // frames with 1 to 4 (a flow field has 2) have kernels here; anything else must not be reinterpreted as bytes
    const bool u8 = frame->type == FrameType::U8 && (ch == 1 || ch == 3 || ch == 4);
    const bool f32 = frame->type == FrameType::F32 && ch >= 1 && ch <= 4;
    if (!u8 && !f32) {
      char msg[160];
      snprintf(msg, sizeof msg, "Resize (B200): %s frames with %d channels are not implemented (U8 with 1, 3 or 4 channels, F32 with 1 to 4)",
               frame_type_name(frame->type), ch);
      STB_FATAL(msg);
    }
    FrameInfo info(target_height, target_width, ch, frame->type);
    std::vector<Frame*> output_frames = new_frames(device_, info, input_count);
    src_.resize(input_count);
    dst_.resize(input_count);
    for (i32 i = 0; i < input_count; ++i) {
      src_[i] = frame_col[i].as_const_frame()->data;
      dst_[i] = output_frames[i]->data;
    }
    if (u8) {
      STB_CHECK(stb_resize_u8(src_.data(), input_count, frame->width(), frame->height(), ch, dst_.data(), target_width,
                              target_height, interp_, stream_));
    } else {
      std::vector<const float*> fs(input_count);
      std::vector<float*> fd(input_count);
      for (i32 i = 0; i < input_count; ++i) {
        fs[i] = reinterpret_cast<const float*>(src_[i]);
        fd[i] = reinterpret_cast<float*>(dst_[i]);
      }
      STB_CHECK(stb_resize_f32(fs.data(), input_count, frame->width(), frame->height(), ch, fd.data(), target_width,
                               target_height, interp_, stream_));
    }
    for (i32 i = 0; i < input_count; ++i) insert_frame(output_columns[0], output_frames[i]);
    CU_CHECK(cudaStreamSynchronize(stream_));
  }

 private:
  DeviceHandle device_;
  cudaStream_t stream_;
  ResizeArgsLite args_;
  int interp_ = 0;
  Result valid_;
  std::vector<const uint8_t*> src_;
  std::vector<uint8_t*> dst_;
};

#ifndef STB_SKIP_OP_DECLARATIONS
REGISTER_OP(Resize).frame_input("frame").frame_output("frame");
#endif

REGISTER_KERNEL(Resize, ResizeKernelGPU).device(DeviceType::GPU).batch().num_devices(1);

// test harness hooks (compat build only): run the kernel with serialized args on n host frames of w x h x c elements
#ifdef STB_COMPAT_SHIM
static int shim_resize(FrameType type, const void* h_frames, int n, int w, int h, int c, const uint8_t* args, int args_len,
                       void* h_out, size_t out_capacity, int* out_w, int* out_h, int device_id) {
  KernelConfig cfg;
  cfg.devices.push_back(DeviceHandle{DeviceType::GPU, device_id});
  ResizeKernelGPU k(cfg);
  k.new_stream(std::vector<u8>(args, args + args_len));
  Result r;
  k.validate(&r);
  if (!r.success()) return -4;
  DeviceHandle dev{DeviceType::GPU, device_id};
  FrameInfo info(h, w, c, type);
  std::vector<Frame*> in = new_frames(dev, info, n);
  BatchedElements input(1), output(1);
  for (int i = 0; i < n; ++i) {
    CU_CHECK(cudaMemcpy(in[i]->data, static_cast<const uint8_t*>(h_frames) + (size_t)i * info.size(), info.size(),
                        cudaMemcpyHostToDevice));
    input[0].push_back(Element(in[i]));
  }
  k.execute(input, output);
  int rc = 0;
  if ((int)output[0].size() != n) rc = -2;
  for (int i = 0; i < n && rc == 0; ++i) {
    Frame* f = output[0][i].as_frame();
    *out_w = f->width(); *out_h = f->height();
    if (f->type != type || (size_t)(i + 1) * f->size() > out_capacity) { rc = -3; break; }
    CU_CHECK(cudaMemcpy(static_cast<uint8_t*>(h_out) + (size_t)i * f->size(), f->data, f->size(), cudaMemcpyDeviceToHost));
  }
  if (!output[0].empty()) delete_buffer(dev, output[0][0].as_frame()->data);
  for (auto& e : output[0]) delete e.as_frame();
  delete_buffer(dev, in[0]->data);
  for (Frame* f : in) delete f;
  return rc;
}

extern "C" __attribute__((visibility("default"))) int stb_shim_resize(const uint8_t* h_frames, int n, int w, int h, int c,
                                                                      const uint8_t* args, int args_len, uint8_t* h_out,
                                                                      int out_capacity, int* out_w, int* out_h, int device_id) {
  return shim_resize(FrameType::U8, h_frames, n, w, h, c, args, args_len, h_out, (size_t)out_capacity, out_w, out_h, device_id);
}

// F32 frames; out_capacity counts floats
extern "C" __attribute__((visibility("default"))) int stb_shim_resize_f32(const float* h_frames, int n, int w, int h, int c,
                                                                          const uint8_t* args, int args_len, float* h_out,
                                                                          int out_capacity, int* out_w, int* out_h, int device_id) {
  return shim_resize(FrameType::F32, h_frames, n, w, h, c, args, args_len, h_out, (size_t)out_capacity * sizeof(float),
                     out_w, out_h, device_id);
}
#endif  // STB_COMPAT_SHIM
}  // namespace scanner
