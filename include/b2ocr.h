/*
 * b2ocr.h -- C-ABI of the B200-native drop-in for keras_ocr.pipeline.Pipeline.recognize().
 *
 * The reference (faustomorales/keras-ocr @ 9661d6f) is pure Python and has no FFI of its own:
 * its "device boundary" is two keras.Model.predict() calls (detection.py:779, recognition.py:535)
 * plus OpenCV calls.  Each entry point below replaces one of those call sites; the reference
 * line(s) it stands in for are cited.  INTEGRATION.md shows the ctypes binding a keras-ocr
 * maintainer would add.
 *
 * Conventions
 *   - plain C: pointers + sizes, no torch / C++ types.  Every function returns 0 on success or a
 *     negative b2o_status; b2o_last_error() gives the message.  No C++ exception crosses the ABI.
 *   - "dev" pointers are CUDA device pointers on the context's device, "host" pointers are host
 *     memory.  All work is enqueued on `stream` (a cudaStream_t passed as void*) and is
 *     asynchronous unless stated.  The caller owns every I/O and workspace buffer; the library
 *     owns only the packed weights inside the context.
 *   - images are NHWC uint8 RGB; activations NHWC fp16; score maps NHWC fp32 (text, link).
 *   - there is NO CPU fallback: without a CUDA device every call fails with B2O_ERR_CUDA.
 */
#ifndef B2OCR_H
#define B2OCR_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b2o_ctx b2o_ctx;

typedef enum {
  B2O_OK = 0,
  B2O_ERR_CUDA = -1,       /* CUDA runtime / driver error (message has the detail)            */
  B2O_ERR_ARG = -2,        /* bad argument (NULL, shape, alignment)                           */
  B2O_ERR_WEIGHTS = -3,    /* missing / mis-shaped tensor in b2o_load_*                       */
  B2O_ERR_WORKSPACE = -4,  /* workspace too small                                             */
  B2O_ERR_STATE = -5       /* call needs weights that were not loaded                         */
} b2o_status;

/* Largest CTC class count (len(alphabet) + 1, recognition.py:376-381) the recognizer accepts; the class
 * count itself is read from the shape of "fc_12.kernel" (256, K) at b2o_load_crnn.                */
#define B2O_MAX_CLASSES 1024

/* One named float32 host tensor (row-major) of a checkpoint, in the reference's naming:
 * CRAFT: PyTorch keys of craft_mlt_25k.pth without the "module." prefix (detection.py:428-468);
 * CRNN : Keras layer names of build_model (recognition.py:214-329), Keras layouts.            */
typedef struct {
  const char* name;
  const float* data;
  int32_t ndim;
  int64_t shape[4];
} b2o_tensor;

/* Which convolution engine to use: B2O_CONV_AUTO = tcgen05 wherever the shape allows (the product
 * path), B2O_CONV_SIMT = CUDA-core debug engine used to cross-check the tcgen05 kernels.      */
enum { B2O_CONV_AUTO = 0, B2O_CONV_SIMT = 1, B2O_CONV_TC_GENERIC = 2 /* tcgen05 without halo tiles / fused pool */ };

int b2o_version(void);
int b2o_create(int device, b2o_ctx** out);
void b2o_destroy(b2o_ctx* ctx);
const char* b2o_last_error(const b2o_ctx* ctx);
int b2o_set_conv_engine(b2o_ctx* ctx, int engine);
/* number of kernels this library has launched since creation (bench.py's gpu_launches) */
int64_t b2o_launch_count(const b2o_ctx* ctx);

/* Measurement hook (bench.py's roofline leg): when enabled, every launch of the tensor-core conv
 * kernel is bracketed by CUDA events on its stream; b2o_profile_read sums the kernel time (ms), the
 * algorithmic FLOPs (2*pixels*taps*cin*cout) and the launch count since b2o_profile_enable(1). */
int b2o_profile_enable(b2o_ctx* ctx, int on);
int b2o_profile_read(b2o_ctx* ctx, double* tc_ms, double* tc_flop, int64_t* tc_launches);

/* Detector() / Recognizer() weight loading (detection.py:686-696, recognition.py:382-404).
 * Folds batch-norm, converts to fp16 and packs into the kernels' layouts on the device.      */
int b2o_load_craft(b2o_ctx* ctx, const b2o_tensor* tensors, int n);
int b2o_load_crnn(b2o_ctx* ctx, const b2o_tensor* tensors, int n);

/* Crop geometry of the recognizer, build_model(height, width, rnn_steps_to_discard) (recognition.py:13-23, 214, 328).
 * Crops are height x width; the conv stack's two floor-ing 2x2 max pools leave T = width / 4 time steps of
 * Hf = height / 4 feature rows, so fc_9.kernel is (Hf*512, 128) and stn.dense_a.kernel (T*Hf*32, 64); label rows are
 * T - rnn_steps_to_discard long.  Call it BEFORE b2o_load_crnn, which checks those shapes against it (B2O_ERR_STATE
 * once a CRNN is loaded).  Default 31 x 200, 2 discarded: T = 50, 48-long label rows.  Supported: height 16..64,
 * width 32..800, 0 <= rnn_steps_to_discard < width / 4 (B2O_ERR_ARG otherwise).  The warp, crop-to-input, forward,
 * workspace and tap entry points below follow the context's geometry.                                           */
#define B2O_CRNN_MIN_HEIGHT 16
#define B2O_CRNN_MAX_HEIGHT 64
#define B2O_CRNN_MIN_WIDTH 32
#define B2O_CRNN_MAX_WIDTH 800
int b2o_set_crnn_geometry(b2o_ctx* ctx, int height, int width, int rnn_steps_to_discard);

/* tools.resize_image + tools.pad (tools.py:378-398, 356-375; pipeline.py:44-57), one image:
 * bilinear (OpenCV fixed-point INTER_LINEAR) resize of src (hs x ws x 3) to (hr x wr), written into
 * the top-left of dst image `index` of a (n, hp, wp, 3) batch; the rest is filled with 255.   */
int b2o_resize_pad(b2o_ctx* ctx, const uint8_t* src_dev, int hs, int ws, int hr, int wr,
                   uint8_t* dst_dev, int index, int hp, int wp, void* stream);

/* The same for a batch of n equally sized sources (n,hs,ws,3) in ONE launch (the 4-D ndarray input of
 * pipeline.py:41-42).  gray, when not NULL, also receives cv2.cvtColor(RGB2GRAY) of the padded batch
 * (n,hp,wp) -- recognition.py:510 -- so that the recognizer need not read the batch again.       */
int b2o_resize_pad_batch(b2o_ctx* ctx, const uint8_t* src_dev, int n, int hs, int ws, int hr, int wr,
                         uint8_t* dst_dev, int hp, int wp, uint8_t* gray_dev, void* stream);

/* tools.read for JPEG input (tools.py:19-38: cv2.imread / cv2.imdecode + BGR->RGB) decoded on the GPU by nvJPEG, so
 * that only the compressed file crosses PCIe.  b2o_jpeg_info parses the header (host only); b2o_decode_jpeg writes
 * (height, width, 3) uint8 interleaved RGB at rgb_dev (gray files are expanded to three equal channels, as
 * cv2.imread's default flag does).  nvJPEG is opened with dlopen on first use: B2O_ERR_STATE if the box has none,
 * B2O_ERR_ARG for a stream it refuses (the caller then decodes that file on the host).  Pixels can differ from
 * libjpeg-turbo's (IDCT rounding: <= 4 levels; 4:2:0 chroma upsampling: up to ~25 levels at sharp colour edges, mean < 0.5);
 * tests/test_gpu_parity.py::test_gpu_jpeg_decode states the bounds.                                             */
int b2o_jpeg_info(b2o_ctx* ctx, const uint8_t* data_host, size_t size, int* height, int* width, int* components);
int b2o_decode_jpeg(b2o_ctx* ctx, const uint8_t* data_host, size_t size, uint8_t* rgb_dev, int height, int width,
                    void* stream);

/* cv2.cvtColor(RGB2GRAY) (recognition.py:510) for a whole (n,h,w,3) batch -> (n,h,w).         */
int b2o_rgb_to_gray(b2o_ctx* ctx, const uint8_t* img_dev, int n, int h, int w, uint8_t* gray_dev,
                    void* stream);

/* compute_input + model.predict of Detector.detect (detection.py:34-42, 777-779): CRAFT forward.
 * img: (n,h,w,3) uint8 RGB.  scores: (n, h/2, w/2, 2) float32.                                */
size_t b2o_craft_workspace_bytes(int n, int h, int w);
int b2o_craft_forward(b2o_ctx* ctx, const uint8_t* img_dev, int n, int h, int w, float* scores_dev,
                      void* ws_dev, size_t ws_bytes, void* stream);

/* getBoxes (detection.py:207-287).  scores: (n,hs,ws,2) float32.  Writes, per image i,
 * counts[i] = number of boxes found (may exceed max_boxes: then only the first max_boxes are
 * stored and the caller retries with a larger buffer) and boxes[i][k][4][2] float32 in
 * detector-input pixels, in connected-component label order (= reference order).              */
size_t b2o_boxes_workspace_bytes(int n, int hs, int ws, int max_boxes);
int b2o_get_boxes(b2o_ctx* ctx, const float* scores_dev, int n, int hs, int ws,
                  float detection_threshold, float text_threshold, float link_threshold,
                  int size_threshold, float* boxes_dev, int32_t* counts_dev, int max_boxes,
                  void* ws_dev, size_t ws_bytes, void* stream);

/* The box bookkeeping of recognize_from_boxes (recognition.py:511-521: crops are appended image after
 * image, start_end = running offsets) on the device: the (n,max_boxes,4,2) table of b2o_get_boxes becomes
 * the dense list flat (sum_i min(counts[i],max_boxes), 4, 2) with image_index[k] = image of box k, both
 * sized for n*max_boxes entries by the caller.  Runs without the host knowing the counts, i.e. BEFORE
 * the one synchronisation of the path.                                                          */
int b2o_compact_boxes(b2o_ctx* ctx, const float* boxes_dev, const int32_t* counts_dev, int n, int max_boxes,
                      float* flat_dev, int32_t* image_index_dev, void* stream);

/* tools.warpBox over box groups (recognition.py:506-519; tools.py:61-117).  boxes: (n_boxes,4,2)
 * float32; image_index[k] selects the gray image of box k.  crops: (n_boxes,height,width) uint8
 * (exactly warpBox's output at the context's crop size, 31 x 200 by default) and, when crnn_in != NULL, the
 * CRNN input (n_boxes,width,height) fp16 = crop/255 after Permute((2,1,3)) and the axis flip of
 * recognition.py:215-216.                                                                      */
int b2o_warp_boxes(b2o_ctx* ctx, const uint8_t* gray_dev, int n, int h, int w,
                   const float* boxes_dev, const int32_t* image_index_dev, int n_boxes,
                   uint8_t* crops_dev, void* crnn_in_dev, void* stream);

/* The same for a recognizer built with color=True (recognition.py:214, 508-510: crops are cut from the RGB image, no
 * gray conversion): rgb (n,h,w,3) uint8, crops (n_boxes,height,width,3) uint8, crnn_in (n_boxes,width,height,3) fp16. */
int b2o_warp_boxes_color(b2o_ctx* ctx, const uint8_t* rgb_dev, int n, int h, int w,
                         const float* boxes_dev, const int32_t* image_index_dev, int n_boxes,
                         uint8_t* crops_dev, void* crnn_in_dev, void* stream);

/* prediction_model.predict (recognition.py:535; graph 214-333): CRNN + STN + BiLSTM + greedy CTC.
 * crnn_in: (b,width,height) fp16 from b2o_warp_boxes (or b2o_crops_to_input).  labels: (b,T-discard) int32
 * ((b,48) at the default geometry), merged + blank-free, padded with -1 -- the tensor recognize_from_boxes
 * iterates (527-534).  b2o_crnn_workspace_bytes has no context and sizes the default 31 x 200 geometry;
 * b2o_crnn_workspace_bytes_for sizes the context's.                                                          */
size_t b2o_crnn_workspace_bytes(int b);
size_t b2o_crnn_workspace_bytes_for(const b2o_ctx* ctx, int b);
/* crops (b,height,width) uint8 -> (b,width,height) fp16 (the layout b2o_warp_boxes writes to crnn_in).        */
int b2o_crops_to_input(b2o_ctx* ctx, const uint8_t* crops_dev, int b, void* crnn_in_dev, void* stream);
/* crops (b,height,width,3) uint8 -> (b,width,height,3) fp16 for a color=True recognizer (conv_1.kernel of shape
 * (3,3,3,64)); b2o_crnn_forward then takes that 3-channel input.                                              */
int b2o_crops_to_input_color(b2o_ctx* ctx, const uint8_t* crops_dev, int b, void* crnn_in_dev, void* stream);
/* Recognizer.recognize's preparation (recognition.py:467-489: tools.fit(cval=0) to the context's crop size, then
 * cv2.cvtColor for a gray model) for b RGB crops of any size at once.  srcs_dev: device array of b device pointers,
 * crop k being (sh,sw,3) uint8, contiguous; crops may live in one staging buffer or in separate allocations.
 * dims_dev: b x (sh, sw, rh, rw) int32, where (rh, rw) is the resize size tools.fit picks (tools.fit_plan), and
 * (rh, rw) = (sh, sw) when it does not resize; a row with a non-positive entry gives an all-zero crop.  crnn_in:
 * (b,width,height) fp16 -- (b,width,height,3) when the loaded CRNN takes RGB crops -- in the layout of
 * b2o_crops_to_input; crops_dev (nullable): the fitted RGB crops (b,height,width,3) uint8, what tools.fit returns.
 * b == 0 is a no-op.                                                                                           */
int b2o_fit_crops(b2o_ctx* ctx, const uint8_t* const* srcs_dev, const int32_t* dims_dev, int b,
                  uint8_t* crops_dev, void* crnn_in_dev, void* stream);
int b2o_crnn_forward(b2o_ctx* ctx, const void* crnn_in_dev, int b, int32_t* labels_dev,
                     void* ws_dev, size_t ws_bytes, void* stream);

/* Result records of Pipeline.recognize for the multi-GPU gather (pipeline.py:66-75; SURVEY.md 8(e)): one
 * fixed-size float32 row per image = [count][rec_boxes x (4,2) boxes * inv_scale[i] (tools.adjust_boxes,
 * tools.py:232-260)][rec_boxes x 48 labels as int8, -1 padded], b2o_record_floats(rec_boxes) floats long.
 * boxes/counts as written by b2o_get_boxes, labels (sum counts, 48) int32 as written by b2o_crnn_forward
 * (NULL when no image has a box).  Rows n..rows-1 (a short last shard) get count -1.  The class count
 * must fit int8 (alphabets up to 126 characters).
 * The *_steps forms take the label row length of a recognizer with another crop geometry (T - discard, see
 * b2o_set_crnn_geometry): labels (sum counts, steps) int32; the label area then holds rec_boxes * steps int8 back
 * to back in rec_boxes * ceil(steps / 4) floats, the unused tail bytes -1.  b2o_record_floats and b2o_pack_records
 * are the forms with steps = 48.                                                                 */
size_t b2o_record_floats(int rec_boxes);
size_t b2o_record_floats_steps(int rec_boxes, int steps);
int b2o_pack_records(b2o_ctx* ctx, const float* boxes_dev, const int32_t* counts_dev, const int32_t* labels_dev,
                     const float* inv_scale_dev, int n, int max_boxes, int rows, int rec_boxes,
                     float* records_dev, void* stream);
int b2o_pack_records_steps(b2o_ctx* ctx, const float* boxes_dev, const int32_t* counts_dev, const int32_t* labels_dev,
                           const float* inv_scale_dev, int n, int max_boxes, int rows, int rec_boxes, int steps,
                           float* records_dev, void* stream);

/* Debug / test taps (not on the product path): b2o_set_debug_taps(ctx, 1) makes b2o_crnn_forward also write the
 * fp32 fc_12 outputs ("logits") to its workspace; by default (0) the fused Dense + CTC kernel keeps them in
 * registers and only the labels reach memory.  b2o_crnn_tap copies an intermediate of the last forward pass.
 * b2o_crnn_tap names: "features" (b,T,Hf,512 f16), "theta" (b,6 f32), "warped" (b,T,Hf,512 f16),
 * "fc_9" (b,T,128 f16), "l1" (b,T,128 f16), "l2" (b,T,256 f16), "logits" (b,T-discard,K f32); at the default
 * geometry T = 50, Hf = 7, T-discard = 48 (b2o_set_crnn_geometry).                             */
int b2o_set_debug_taps(b2o_ctx* ctx, int on);
int b2o_crnn_tap(b2o_ctx* ctx, const char* name, const void* ws_dev, int b, void* out_dev,
                 size_t out_bytes, void* stream);

/* One generic convolution through the selected engine (test hook for the conv kernels).
 * x: (n,h,w,cin) fp16, wgt: (cout, k, k, cin) fp32 host, epilogue y = relu?(acc*s1+t1)*s2+t2.
 * out: (n,h,w,cout) fp16.  s2/t2 may be NULL.                                                 */
int b2o_conv2d_test(b2o_ctx* ctx, const void* x_dev, int n, int h, int w, int cin,
                    const float* wgt_host, int cout, int ksize, int dilation,
                    const float* s1_host, const float* t1_host, int relu,
                    const float* s2_host, const float* t2_host, void* out_dev, int engine,
                    void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B2OCR_H */
