/*
 * davo_b200.h -- C ABI of libdavo_b200.so: the B200 (sm_100a) implementation of
 * DAVO's pose-estimation forward path (attention module -> masked frame stack ->
 * dilated PoseNN -> 6-DoF per frame pair).
 *
 * The reference (BassyKuo/DAVO) has no FFI layer: its boundary for this path is
 * the Python class `DAVO` over a TensorFlow session.  Each entry point below
 * names the reference interface it stands in for (paths relative to the
 * reference checkout).  The Python mirror of that class (davo_b200/davo.py)
 * binds these symbols with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions: every function returns 0 on success and a negative davo_status
 * on failure; davo_last_error() then describes it.  A handle is bound to one
 * CUDA device, is not thread-safe, launches only on the caller's stream and
 * never synchronises inside davo_forward.  Device buffers passed in are owned
 * by the caller; weights and activation workspace are owned by the handle.
 * There is no CPU fallback: without a CUDA device every call fails.
 */
#ifndef DAVO_B200_H
#define DAVO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct davo_ctx davo_ctx;

enum davo_status {
  DAVO_OK = 0,
  DAVO_ERR_ARG = -1,        /* bad argument / unsupported configuration */
  DAVO_ERR_CUDA = -2,       /* CUDA runtime or driver error             */
  DAVO_ERR_WEIGHT = -3,     /* unknown / missing / mis-shaped variable  */
  DAVO_ERR_STATE = -4       /* call order (e.g. forward before finalize)*/
};

/* Filled by the version-string parser (davo_b200/version.py), which mirrors
 * reference davo.py:1010-1102 (option groups) and :1117-1450 (attention source
 * and masking chain). */
typedef struct davo_config {
  int32_t H, W;          /* frame size, reference test_kitti_pose.py:22-23 (128, 416)  */
  int32_t max_batch;     /* largest B (samples) a forward call may carry               */
  int32_t posenn;        /* nets/posenn.py, selected at davo.py:1027-1049:
                            0 decouple_sharednet_v0_dilation (:189, headline), 1 couple_sharednet_v0_dilation (:133),
                            2 decouple_net_v0_dilation (:69), 3 couple_net_v0_dilation (:12),
                            4 couple_net_v0 (:257), 5 decouple_net_v0 (:314); 2-5 evaluate a whole sample at once */
  int32_t cnv6_out;      /* "-cnv6_<n>", davo.py:1052-1053: 32, 64, 128 or 256         */
  int32_t in_mode;       /* 0 = v0 RGB only, 1 = v1 RGB+flow, davo.py:1057-1065        */
  int32_t att_src;       /* 0 none, 1 se_flow (davo.py:1175), 2 static (:1390), 3 se_seg (:1304),
                            4 se_rgb -> seg (:1274), 5 se_depth -> seg (:1211),
                            6 se_segflow -> seg (:1341-1372; se_hidden 8 for the "_8" tokens) */
  int32_t att_tgt_ones;  /* target-frame map forced to 1, davo.py:1404-1412, :1393     */
  int32_t mask_mode;     /* 0 off, 1 rgb, 2 all, 3 all(.555), davo.py:1415-1450        */
  int32_t se_act;        /* 0 relu, 1 tanh, 2 leaky_relu(0.2), davo.py:1077-1085       */
  int32_t flow_abs;      /* 0 none, 1 both, 2 h, 3 v, davo.py:1094-1102                */
  int32_t flow_norm;     /* "-norm_flow", davo.py:1088-1091                            */
  int32_t posenn_se;     /* 0 none, 1 insert, 2 skipadd (needs cnv6_out 256), 3 replace, davo.py:1010-1017, posenn.py:225-236 */
  int32_t micro_batch;   /* units (frame pairs; samples for posenn 2-5) per pass of the conv stack; 0 = 256 */
  int32_t depth_norm;    /* att_src 5: 0 depth_i + depth_tgt (davo.py:1109), 1 the same / 80 ("-norm_depth",
                            :1110-1111), 2 the se_disp sources: 1 / depth_i (:1253-1270)            */
  int32_t se_pool;       /* se_flow and se_seg: 0 global mean, 1 gp2x2 (four quadrants, davo.py:1181-1192, 1317),
                            2 / 3 / 4 spatial pyramid [2,1] / [2] / [8,6,4] (davo.py:1193-1210, 1323-1340) */
  int32_t se_hidden;     /* width of the SE bottleneck; 0 = the source's default (8; se_seg 19)  */
  int32_t pixel_map;     /* 1: the se_block sources whose map is reduce_sum(input * excitation) per pixel rather
                            than a class weight gathered by label: att_src 4 -se_rgb[_wo_tgt] (davo.py:1293-1303),
                            5 -se_depth[_wo_tgt] / -se_disp[_wo_tgt] (:1228-1245, 1271-1292), 6 -se_mixSegFlow
                            (:1375-1379); 2 (att_src 5 only): depth term AND SE flow, -se_mixDepthFlow /
                            -se_mixDispFlow (:1157-1174); shared nets only                           */
  int32_t depth_split;   /* 1: -se_flow_on_depthseg_seplayers (davo.py:1136-1154), att_src 1 only: two SEs on the flow,
                            "se_flow_near" / "se_flow_far"; a pixel takes its class weight from the near table where
                            its depth is below the variable se_flow/depth_threshold, else from the far table; reads
                            input_depth; shared nets only                                            */
  int32_t flow_f16;      /* 0 (default): the optical flow is read as the float32 it is given in, like the reference's
                            graph (davo.py:978-982; the SE pooling, attention_module.py:66, averages float32 values).
                            1: opt-in transport narrowing -- every flow value is rounded to IEEE binary16 when read (11
                            significant bits, what a TF32 conv operand keeps; the SE pooling then averages the rounded
                            values: class weights move by <= 1.5e-5 relative, poses by ~2e-8), on BOTH entry points, so
                            that davo_forward_host may move the flow over PCIe as binary16 with results bit-identical
                            to davo_forward in the same mode                                         */
  int32_t batch_norm;    /* "-batch_norm" (davo.py:1453, posenn.py:206): slim.batch_norm on every conv except pred, and --
                            because the reference passes no normalizer_params -- with slim's default is_training=True at
                            test time: each layer is normalised with the mean / biased variance of the batch of its
                            PoseNN call (the shared nets make two calls: all tgt->src0 pairs, all tgt->src1 pairs);
                            variables <conv>/BatchNorm/beta instead of <conv>/biases.  The poses therefore depend on
                            which samples share a call: the whole batch must fit one pass (2*B, or B for posenn 2-5,
                            <= micro_batch), every pair is computed (DAVO_PAIRS_ALL) and only the device entry points
                            take it                                                                  */
} davo_config;

/* Stands in for DAVO.__init__ + DAVO.setup_inference (reference davo.py:31-33,
 * 1533-1551): fixes the variant, frame size and batch, allocates workspaces. */
int davo_create(const davo_config* cfg, int device, davo_ctx** out);

/* Stands in for tf.train.Saver(...).restore (reference test_kitti_pose.py:129-131),
 * one variable at a time, keyed by TF variable name.  Conv kernels are HWIO,
 * dense kernels [in, out], as TF stores them; rank 0 is a scalar variable.  `host` is host memory. */
int davo_set_weight(davo_ctx*, const char* tf_var_name, const float* host,
                    const int64_t* shape, int rank);

/* Checks every variable of the variant was supplied, repacks to the kernels'
 * K-major TF32 layout and uploads. */
int davo_finalize_weights(davo_ctx*);

/* Stands in for DAVO.inference(sess, mode='pose') = one sess.run of pred_poses
 * (reference davo.py:1553-1569) on B <= max_batch samples.
 *   img_u8   device, uint8  [B, H, 3W, 3]   (src0 | tgt | src1 along width)
 *   flow     device, float  [B, 4, H, W, 2] (only [:,0:2] are read, davo.py:978-982); read as float32
 *            unless davo_config.flow_f16 = 1 (then rounded to binary16 when read; values with no finite
 *            half, |x| >= 65520 or NaN, are used as they are)
 *   seg      device, float  [B, 3, H, W, 1] ([src0, tgt, src1], davo.py:1000-1004)
 *   depth    device, float  [B, 3, H, W, 1] ([src0, tgt, src1], davo.py:991-996): read by the
 *            se_depth variants only (att_src 5); NULL otherwise
 *   pose_out device, float  [B, 2, 6]: rows [tgt->src0, tgt->src1],
 *            cols [rz, ry, rx, tx, ty, tz] (nets/posenn.py:193, davo.py:1458)
 * Asynchronous on `cuda_stream` (a cudaStream_t; NULL = default stream). */
int davo_forward(davo_ctx*, int B, const uint8_t* img_u8, const float* flow,
                 const float* seg, const float* depth, float* pose_out,
                 void* cuda_stream);

/* Which frame pairs of the batch are computed.  The reference's consumer of pred_poses,
 * test_kitti_pose.py:136-153, composes only pose[s][1] (tgt->src1) of every sample plus
 * pose[0][0] (tgt->src0) of the first sample of a sequence (:143-145): the other half of the
 * graph's work is discarded.  The TRAJECTORY selections compute exactly what that loop reads;
 * the rows of pose_out that are not computed are set to zero.  The output file is identical. */
enum {
  DAVO_PAIRS_ALL = 0,               /* [B,2,6], as sess.run(pred_poses)            */
  DAVO_PAIRS_TRAJECTORY = 1,        /* pose[s][1] for every s                      */
  DAVO_PAIRS_TRAJECTORY_FIRST = 2   /* ... and pose[0][0]: the chunk that opens a sequence */
};
int davo_forward_pairs(davo_ctx*, int B, int pairs, const uint8_t* img_u8, const float* flow,
                       const float* seg, const float* depth, float* pose_out,
                       void* cuda_stream);
int davo_forward_host_pairs(davo_ctx*, int B, int pairs, const uint8_t* img_u8, const float* flow,
                            const float* seg, const float* depth, float* pose_out,
                            void* cuda_stream);

/* DAVO.inference(sess, mode='feature') (reference davo.py:1553-1564): the poses plus what the
 * reference fetches for visualisation (consumer generate_feature_map.py:183-380).  DEVICE buffers,
 * any of them NULL to skip it; frame order of the [3]-lists is the reference's: tgt, src0, src1.
 * The batch must fit one pass of the conv stack (2*B, or B for posenn 2-5, <= micro_batch). */
typedef struct {
  float*   image;         /* [3][B,H,W,3]   tgt_images: the frames in [-1,1]            (davo.py:967-971)  */
  float*   attention;     /* [3][B,H,W,1]   masks['attention'], after the target override (:1404-1412, 1467) */
  float*   masked_image;  /* [3][B,H,W,3]   masks['image']: input_images[f][..., :3]     (:1470-1474)       */
  float*   seg_19;        /* [3][B,H,W,19]  one_hot(int32(seglabel), 19)                 (:1115)            */
  uint8_t* seg_color;     /* [3][B,H,W,3]   segs: Cityscapes colouring of the labels     (:1005)            */
  uint8_t* flow_color;    /* [2][B,H,W,3]   flows: Middlebury colouring of flow[:,0:2]   (:988-989)         */
  float*   cnv6_rot;      /* [B,H,W,cnv6_out] features['rot']: cnv6 of the last PoseNN call (tgt->src1 for the
                             shared nets), resize_bilinear to HxW                        (:1456-1465)       */
  float*   cnv6_trans;    /* [B,H,W,cnv6_out] features['trans'] (the same tensor as rot for the couple nets) */
} davo_features;
int davo_forward_features(davo_ctx*, int B, const uint8_t* img_u8, const float* flow,
                          const float* seg, const float* depth, float* pose_out,
                          const davo_features* out, void* cuda_stream);

/* Same call with HOST buffers (pinned for overlap; pageable works): the end-to-end
 * form of `sess.run` with fed numpy arrays (reference davo.py:1568).  The batch is
 * streamed in micro-batch chunks, the host->device copy of chunk i+1 overlapping
 * the compute of chunk i; only the planes the graph reads are copied (flow[:,0:2],
 * and seg[:,{0,2}] when the target map is ones), the labels as bytes (lossless: the graph casts them
 * to int32, davo.py:1115) and -- only with davo_config.flow_f16 = 1, on a host with >= 16 hardware
 * threads that this process does not share with other ranks -- three quarters of the flow as binary16,
 * both narrowed by a small CPU thread pool inside the call (DAVO_B200_HOST_SEG8 / _FLOW16 /
 * _FLOW16_FRAC / _THREADS override).  Results are bit-identical to the device entry point of the
 * same configuration either way.  Poses are copied back and the stream synchronised
 * before returning. */
int davo_forward_host(davo_ctx*, int B, const uint8_t* img_u8, const float* flow,
                      const float* seg, const float* depth, float* pose_out,
                      void* cuda_stream);

/* The same call for a caller that already holds the inputs in compact form (its own loader decoded the labels to
 * bytes and keeps the flow in half precision): nothing is converted on the CPU, the planes go from the caller's
 * (ideally pinned) memory straight to the device, 1.06 MB per sample instead of 1.44 MB.
 *   flow_f16  host, IEEE binary16 [B, 2, H, W, 2]: the two planes the graph reads (flow[:,0:2], davo.py:978-982);
 *             widened exactly, so the result equals davo_forward on the widened values in either flow_f16 mode
 *   seg_u8    host, uint8 [B, 3, H, W]: tf.cast(seglabel, int32) (davo.py:1115) clamped to a byte, any value
 *             outside 0..18 meaning "no class" (255 by convention)
 * `pairs` as in davo_forward_pairs.  This is an EXTENSION of the reference's input contract (which feeds float32
 * flow and labels, test_kitti_pose.py:104-114); bench.py reports it as a separate, labelled end-to-end number. */
int davo_forward_host_compact(davo_ctx*, int B, int pairs, const uint8_t* img_u8, const uint16_t* flow_f16,
                              const uint8_t* seg_u8, const float* depth, float* pose_out, void* cuda_stream);

/* Asynchronous forms of the two host entry points: the call returns as soon as its copies and launches are queued
 * (chunk by chunk, as above), so the copies of the NEXT batch run under the compute of this one -- the reference gets
 * the same overlap from tf.data's prefetch in front of sess.run.  `pose_out` must be page-locked and stay valid until
 * davo_host_wait(ctx, *ticket) returns; calls complete in issue order; the input buffers may be reused as soon as the
 * call returns only if they are not written before davo_host_wait (the DMA engine reads them in place).  At most 8
 * tickets are remembered: waiting for an older one waits for a later call, which implies it. */
int davo_forward_host_pairs_async(davo_ctx*, int B, int pairs, const uint8_t* img_u8, const float* flow,
                                  const float* seg, const float* depth, float* pose_out, void* cuda_stream,
                                  long long* ticket);
int davo_forward_host_compact_async(davo_ctx*, int B, int pairs, const uint8_t* img_u8, const uint16_t* flow_f16,
                                    const uint8_t* seg_u8, const float* depth, float* pose_out, void* cuda_stream,
                                    long long* ticket);
int davo_host_wait(davo_ctx*, long long ticket);

/* --- frame-sequence inputs ---
 * A camera stream or a video as it comes: N >= 3 frames and the flow between neighbours, each frame sent once
 * instead of once per sample that holds it.  Sample s (0 <= s < N-2) is frames (s, s+1, s+2) in the roles
 * (src0, tgt, src1); poses land in pose_out [N-2,2,6] with the rows, columns and pair selections (`pairs`) of
 * davo_forward_pairs.  Every buffer is contiguous and 16-byte aligned:
 *   img       uint8 [N,H,W,3]
 *   flow_fwd  float [N-1,H,W,2]  entry i: flow from frame i to frame i+1   (sample s: flow[:,0] = flow_fwd[s])
 *   flow_bwd  float [N-1,H,W,2]  entry i: flow from frame i+1 to frame i   (sample s: flow[:,1] = flow_bwd[s+1])
 *   seg       float [N,H,W,1]    labels as in davo_forward; NULL for variants without attention source
 *   depth     float [N,H,W,1]    the depth sources only, otherwise NULL
 * flow_fwd may be NULL for the shared nets under DAVO_PAIRS_TRAJECTORY (only flow_fwd[0] is read under
 * DAVO_PAIRS_TRAJECTORY_FIRST); both may be NULL for variants that read no flow.  The poses are bit-identical to
 * davo_forward_pairs on the triplet batch built from the same frames (davo_b200.sequence_to_triplets).  A long
 * sequence continues with a call that starts two frames before the previous one ended: only those two frames are
 * sent again, no flow is.  Argument errors (N < 3, N-2 > max_batch, a NULL input the variant and selection read, a
 * misaligned buffer) return DAVO_ERR_ARG with a message naming the input.
 *
 * davo_forward_sequence: device buffers, as davo_forward_pairs (-batch_norm included: one pass, DAVO_PAIRS_ALL).
 * davo_forward_sequence_host: host buffers, as davo_forward_host_pairs: chunked, copies overlapping compute, labels
 *   (and with flow_f16 = 1 the flow) narrowed on the CPU.  Each frame plane and flow entry crosses PCIe at most once
 *   per call, and those that no computed pair reads are not copied (davo_last_host_copy_bytes counts them).
 *   ticket == NULL: blocks until the poses are in pose_out; otherwise the asynchronous form of
 *   davo_forward_host_pairs_async, waited for with davo_host_wait. */
int davo_forward_sequence(davo_ctx*, int n_frames, int pairs, const uint8_t* img_u8, const float* flow_fwd,
                          const float* flow_bwd, const float* seg, const float* depth, float* pose_out,
                          void* cuda_stream);
int davo_forward_sequence_host(davo_ctx*, int n_frames, int pairs, const uint8_t* img_u8, const float* flow_fwd,
                               const float* flow_bwd, const float* seg, const float* depth, float* pose_out,
                               void* cuda_stream, long long* ticket);

/* --- online odometry sessions ---
 * A camera loop: push frames as they arrive, get each frame's absolute pose, composed on the device.  A session
 * belongs to one handle and takes one sequence in order, k >= 1 new frames per push.  With f0 frames pushed so far, a
 * push carries frames f0 .. f0+k-1 in the layouts of davo_forward_sequence:
 *   img       uint8 [k,H,W,3];  seg float [k,H,W,1] (NULL for variants without attention source);  depth float
 *             [k,H,W,1] (depth sources only)
 *   flow_fwd, flow_bwd  float [k',H,W,2], k' = k (k-1 on the first push): entry j is the sequence's flow entry
 *             f0-1+j (j on the first push), i.e. a push is img[a:b], flow[a-1:b-1] of a whole-sequence call
 *             (flow[0:b-1] for the first).  A flow no computed pair reads may be NULL, as in davo_forward_sequence.
 * It computes every sample whose last frame is new (s+2 in [f0, f0+k): none for a first push of 1 or 2 frames):
 *   pose_out  float [n_samples,2,6]  rows and columns of davo_forward_pairs; under DAVO_PAIRS_TRAJECTORY only
 *             pose[s][1], plus pose[0][0] for sample 0 (the trajectory reads it)
 *   traj_out  double [n_traj,4,4]    absolute poses of the frames whose pose became known: frames 0, 1, 2 with
 *             sample 0 (P_0 = I, P_1 = T(pose[0][0])), then frame s+2 for sample s, P_{s+2} = P_{s+1} . inv(T(pose[s][1]))
 *             -- the loop of reference test_kitti_pose.py:136-149 with T = pose_vec2mat in fp32, chained in fp64 in
 *             frame order, so the bits do not depend on how the stream is cut into pushes
 * The poses equal davo_forward_sequence over the whole sequence (DAVO_PAIRS_TRAJECTORY_FIRST or DAVO_PAIRS_ALL) bit
 * for bit for every cut; each frame, label plane, depth plane and flow entry a computed pair reads is sent once over
 * the whole stream (davo_last_host_copy_bytes counts a host push's bytes).  The session keeps the last two frames, the
 * last flow_fwd entry when a later sample reads it and the last absolute pose in buffers of its own: sessions on one
 * handle are independent, and other calls on the handle may run between pushes.
 *
 * davo_odometry_create: max_push = most frames per push (1..max_batch); pairs = DAVO_PAIRS_TRAJECTORY or
 *   DAVO_PAIRS_ALL; host_inputs = 1: pushes pass host buffers and get host results (chunked, copies under compute,
 *   CPU narrowing, as davo_forward_sequence_host); 0: device buffers in, device results out, asynchronous on
 *   cuda_stream.  -batch_norm is refused (its poses depend on which samples share a call).
 * davo_odometry_push: *n_samples / *n_traj (either may be NULL) receive the counts.  Host sessions: ticket == NULL
 *   blocks until the results are in pose_out / traj_out; otherwise they must be page-locked, the call returns once
 *   queued, and davo_host_wait(ctx, *ticket) waits for it.  Argument errors (k outside 1..max_push, a NULL input the
 *   variant and selection read, a misaligned buffer, a ticket on a device session, a destroyed session) return
 *   DAVO_ERR_ARG with a message naming the input (davo_last_error(NULL) for a destroyed session).
 * davo_odometry_reset: the next push is frame 0 of a new sequence (P_0 = I).
 * davo_odometry_frames: frames pushed, and frames whose absolute pose has been written.
 * davo_odometry_destroy: waits for the device and frees the session; davo_destroy destroys the handle's sessions. */
typedef struct davo_odometry davo_odometry;
int davo_odometry_create(davo_ctx*, int max_push, int pairs, int host_inputs, davo_odometry** out);
int davo_odometry_push(davo_odometry*, int k, const uint8_t* img, const float* flow_fwd, const float* flow_bwd,
                       const float* seg, const float* depth, float* pose_out, double* traj_out, int* n_samples,
                       int* n_traj, void* cuda_stream, long long* ticket);
/* davo_odometry_push_many: one push on each of n device sessions (host_inputs = 0) of one handle, in one forward pass
 *   -- many cameras, a few frames each, at the same time.  Every array has n entries and lives in host memory; the
 *   pointers it holds are device buffers.  Entry i is what davo_odometry_push(sessions[i], k[i], img[i], flow_fwd[i],
 *   flow_bwd[i], seg[i], depth[i], pose_out[i], traj_out[i], &n_samples[i], &n_traj[i], cuda_stream, NULL) takes:
 *   the same shapes, NULL rules, 16-byte alignment and output rows.  flow_fwd, flow_bwd, seg, depth, n_samples and
 *   n_traj may be NULL as whole arrays when no entry needs them.
 *   The results are bit-identical to pushing each session alone with davo_odometry_push, in array order: pose_out
 *   (with the zero rows of trajectory mode), traj_out, the counts and every later push on those sessions, single or
 *   batched.  Sessions may be in any state (first push, mid-stream, just reset), and trajectory and all-mode sessions
 *   may be mixed; the handle's other sessions are untouched.  Asynchronous on cuda_stream, no synchronisation; the
 *   number of kernel launches does not depend on n.  The first batched push on a handle allocates a staging batch of
 *   max_batch samples, freed with the handle.
 *   Argument errors return DAVO_ERR_ARG with a message naming the input and the session index: n < 1; a NULL or
 *   destroyed session (davo_last_error(NULL)); a session given twice; a host session; sessions of two handles; k[i]
 *   outside 1..max_push; more than max_batch samples in all; a NULL or misaligned buffer entry i reads.  A refused
 *   call enqueues nothing and changes no session. */
int davo_odometry_push_many(int n, davo_odometry* const* sessions, const int* k, const uint8_t* const* img,
                            const float* const* flow_fwd, const float* const* flow_bwd, const float* const* seg,
                            const float* const* depth, float* const* pose_out, double* const* traj_out,
                            int* n_samples, int* n_traj, void* cuda_stream);
/* davo_odometry_push_many_host: one push on each of n host sessions (host_inputs = 1) of one handle, in one forward
 *   pass -- many cameras whose frames arrive in host memory.  Entry i is what davo_odometry_push(sessions[i], k[i],
 *   img[i], ..., cuda_stream, ticket) takes on a host session: the same host buffers, shapes, NULL rules, 16-byte
 *   alignment and output rows; whole arrays may be NULL as for davo_odometry_push_many.  The results are bit-identical
 *   to pushing each session alone with davo_odometry_push, in array order (pose_out, traj_out, the counts and every
 *   later push, single or batched); sessions may be in any state and either pair mode, and single and batched host
 *   pushes mix freely on the same sessions.  ticket == NULL: blocks until every session's results are in host memory;
 *   otherwise the outputs must be page-locked, the call returns once everything is queued, davo_host_wait(ctx, *ticket)
 *   waits for it, and the inputs must not be written before then.  Each new frame, label plane, depth plane and flow
 *   entry that some computed pair of its stream reads is copied once, as by the single push (labels narrowed to bytes
 *   on the CPU unless DAVO_B200_HOST_SEG8=0; the flow as float32); davo_last_host_copy_bytes reports the call's data
 *   bytes, with the default configuration the sum of what the same pushes made one by one report.  The kernel launches
 *   do not depend on n; the copies are per session.  The first call allocates two arrivals sets that grow on demand,
 *   freed with the handle.
 *   Argument errors return DAVO_ERR_ARG with a message naming the input and the session index, as for
 *   davo_odometry_push_many; a device session is refused (davo_odometry_push_many takes it).  A refused call enqueues
 *   nothing and changes no session. */
int davo_odometry_push_many_host(int n, davo_odometry* const* sessions, const int* k, const uint8_t* const* img,
                                 const float* const* flow_fwd, const float* const* flow_bwd, const float* const* seg,
                                 const float* const* depth, float* const* pose_out, double* const* traj_out,
                                 int* n_samples, int* n_traj, void* cuda_stream, long long* ticket);
int davo_odometry_reset(davo_odometry*);
int davo_odometry_frames(const davo_odometry*, long long* pushed, long long* posed);
void davo_odometry_destroy(davo_odometry*);
/* davo_odometry_move: re-homes a live session onto handle `dst`, which may be on another device -- to rebalance
 *   cameras over the GPUs of a box, or to drain a handle without restarting its cameras' trajectories.  The session
 *   pointer stays valid; afterwards it belongs to dst (davo_destroy(dst) destroys it, davo_destroy of the old handle no
 *   longer does) and takes pushes, single or batched with dst's other sessions, of dst.  Every later push gives the
 *   bits it would have given without the move: pose_out, traj_out, the counts, davo_odometry_frames, and the host to
 *   device bytes of a host push.  The counts and the carried state (last two frames with their labels and depth, the
 *   last flow_fwd entry when a later sample reads it, the last absolute pose) are copied with cudaMemcpyPeerAsync, which
 *   needs no peer access (none is enabled); the frame sets and per-push buffers are allocated again on dst at the
 *   session's max_push, and the old buffers are freed.
 *   Synchronises: first waits for all work on the session's device (as davo_odometry_destroy), then returns once the
 *   copies are complete.  Tickets issued on the old handle before the move stay valid there.
 *   A move to the session's own handle returns 0 and does nothing.  Refused with DAVO_ERR_ARG, changing nothing, and a
 *   message on the session's handle (davo_last_error(NULL) for a NULL or destroyed session) naming the reason: a NULL
 *   or destroyed session; dst NULL; a davo_config field other than max_batch that differs (named); the session's
 *   max_push above dst's max_batch; weights not finalized on either handle; different weights (a digest of the values
 *   davo_finalize_weights was given); a different DAVO_B200_WEIGHT_ROUNDING or conv implementation; for a host session
 *   with labels, a different DAVO_B200_HOST_SEG8. */
int davo_odometry_move(davo_odometry*, davo_ctx* dst);

/* Binds the calling thread (and the threads it creates afterwards: the handle's conversion pool, the caller's
 * loader threads) to the CPUs of the NUMA node the handle's GPU hangs off (/sys/bus/pci/devices/<id>/numa_node,
 * local_cpulist), so that pinned staging allocated afterwards is first-touched next to the GPU and the conversion
 * threads read local memory.  Opt-in (it changes the caller's CPU affinity); a host without NUMA information or
 * with one node is left as it is.  Returns the node (>= 0), or -1 when nothing was bound. */
int davo_bind_host_numa(davo_ctx*);

/* Test / mode='feature' access to what the last davo_forward left in the
 * workspace for frame pair `pair` (= 2*sample + source index) of the LAST
 * micro-batch: "att_weights" [19] (slot 0 below; the static table; ones
 * without an attention source), "packed" [H,W,packed_c] (the cnv1 input:
 * packed_c = 8 for the 8-channel layout, 16 for the 16-channel and the
 * whole-sample layouts), "cnv1".."cnv5", "cnv6" [h,w,2*cnv6_out]
 * (rotation | translation), "cnv7_sum" [2,256] (the head's partial sums
 * added in the head's order), "cnv7" where it is stored (-batch_norm: the
 * plain conv sums), "se5_scale" [branches,256] (the excitation of -se_insert
 * / -se_skipadd / -se_replace).
 * "att_weights:<k>" is slot k of the unit's attention weights: 19 class
 * weights, or the excitation of a per-pixel source (its SE input's channels:
 * 3 rgb, 1 depth term, 3 depth term + SE flow, 21 one-hot + SE flow).  Slots:
 *   frame-pair units (shared nets): 0 the source frame, 1 the target (or,
 *     under -se_flow_on_depthseg_seplayers, the "far" table of the source);
 *   sample units (non-shared nets): 0 src0, 1 src1, 2 the target; with the
 *     depth split (0, 1) src0 near / far and (2, 3) src1 near / far.
 * Static variants give the static table for every frame that has a map.  A
 * slot the variant does not compute is refused (DAVO_ERR_ARG).
 * Per conv layer "<layer>" also takes a suffix:
 *   "<layer>"          the map [h,w,C]; an odd map stored with an even pitch
 *                      comes back without its zero pad row / column;
 *   "<layer>:pitched"  the whole stored buffer [h_p,w_p,C];
 *   "<layer>:in"       the input the layer's kernel reads [h_in_p,w_in_p,C_in];
 *   "<layer>:w<g>"     the TF32 weights of group g the kernel's weight pack was
 *                      built from, HWIO over the group's input channels
 *                      [k,k,C_in_g,C_out_g] (zero where no weight is read);
 *   "<layer>:b"        the bias [groups*C_out_g] (-batch_norm: beta);
 *   "<layer>:plan"     the plan the last pass ran: orient (0 pixels-on-M,
 *                      1 channels-on-M), pixels per tile, widened G, widened
 *                      runs per tile row, cm staged, cm cluster, strips,
 *                      m-blocks, groups, raw (-batch_norm), epilogue (0 store,
 *                      1 sum), C_out_g, weights resident, fused front end.
 * Copies to HOST memory `out` (capacity `cap` floats); writes the element
 * count to *n, or the count needed when `cap` is too small.  Synchronises. */
int davo_get_intermediate(davo_ctx*, const char* name, int pair, float* out,
                          int64_t cap, int64_t* n);

/* Bytes the last host entry point (davo_forward_host*, davo_forward_sequence_host) moved host->device and
 * device->host. */
int davo_last_host_copy_bytes(const davo_ctx*, long long* h2d, long long* d2h);

/* Number of kernel launches the last davo_forward issued. */
int davo_last_launch_count(const davo_ctx*);

/* Times each kernel of the last forward's first micro-batch in isolation:
 * re-launches it `iters` times on `cuda_stream` between CUDA events and returns
 * mean milliseconds in ms_out[9] = {front end (pool + pack), cnv1..cnv7, head}.
 * *npairs_out receives the frame pairs per launch.  Synchronises. */
int davo_profile_layers(davo_ctx*, int iters, float* ms_out, int* npairs_out,
                        void* cuda_stream);

/* Test hook: 0 = tcgen05 implicit GEMM (the product path), 1 = plain fp32
 * direct convolution on CUDA cores, used only to cross-check the tensor-core
 * path on the GPU. */
int davo_debug_set_conv_impl(davo_ctx*, int impl);
/* Test hook, CPU only: the float32 -> IEEE binary16 conversion the host entry point applies to the
 * flow planes before they cross PCIe (portable != 0: the scalar path instead of F16C).  Returns 0,
 * or 1 when some value has no finite half (|x| >= 65520, NaN): such a chunk is sent as float32. */
int davo_debug_flows_to_half(const float* src, uint16_t* dst, long long n, int portable);
/* Test hook, CPU only: the float32 label -> byte conversion of the host entry point (tf.cast(label, int32),
 * reference davo.py:1115, then "outside 0..18 -> 255 = an all-zero one_hot row", NaN included like the device
 * conversion); portable != 0: the scalar path instead of AVX2 / SSE2. */
int davo_debug_labels_to_bytes(const float* src, uint8_t* dst, long long n, int portable);

/* --- multi-GPU: one process and one handle per GPU, samples sharded by rank, one collective ---
 * The reference is single-process (test_kitti_pose.py:133-153); sharding its sample list by rank
 * needs one exchange, the all-gather of the [n_local,2,6] pose blocks before the sequential
 * composition on the host.  NCCL is bound at run time (libnccl.so.2; DAVO_B200_NCCL_LIB overrides).
 *
 * davo_comm_unique_id: rank 0 fills 128 bytes (an ncclUniqueId) and hands them to the other ranks
 *   by whatever side channel the host has (torch.distributed store, MPI, a file).
 * davo_comm_create: collective over all ranks; builds the handle's own communicator on its device.
 * davo_allgather_poses: enqueues on `cuda_stream` the gather of `n_local` samples (n_local*12
 *   floats, the same on every rank -- pad the last shard as utils/common_utils.py:8-13 pads a
 *   batch); rank r's block lands at all + r*n_local*12.  `nccl_comm` is an ncclComm_t the host
 *   already owns, or NULL for the handle's communicator; with neither, the world is one rank and
 *   the call is a device copy.  No host synchronisation. */
#define DAVO_COMM_ID_BYTES 128
int davo_comm_unique_id(void* id128);
int davo_comm_create(davo_ctx*, const void* id128, int rank, int world);
int davo_comm_world(const davo_ctx*, int* rank, int* world);
int davo_allgather_poses(davo_ctx*, void* nccl_comm, const float* local_dev, int n_local,
                         float* all_dev, void* cuda_stream);

/* --- on-device trajectory composition and KITTI evaluation (SURVEY 8f-4) ---
 * davo_compose_trajectory stands in for the host loop of reference test_kitti_pose.py:136-149 at its shipped
 * --batch_size 1: rel = [T(pose[0,0])] + [inv(T(pose[s,1])) for every sample s] with T = pose_vec2mat
 * (utils/geo_utils.py:12-63, 93-119, fp32 like the TF graph), P_0 = I, P_{i+1} = P_i . rel_i in fp64 -- as a
 * blocked parallel prefix product instead of a sequential chain.
 *   poses_dev  device, float  [n_samples, 2, 6] (what davo_forward / davo_allgather_poses wrote)
 *   traj_dev   device, double [n_samples + 2, 4, 4] absolute poses, row-major
 * davo_kitti_errors stands in for calcSequenceErrors + saveStats of the reference's KITTI devkit
 * (kitti_benchmark/cpp/test_odometry_all.cpp:44-125, 395-404): segment lengths 100..800 m, first frames every 10
 * frames, distances accumulated in float in frame order as the devkit does.
 *   gt_dev, res_dev  device, double [n_frames, 4, 4]
 *   seg_dev          device, davo_kitti_segment [ceil(n_frames / 10) * 8] or NULL; last_frame = -1: the sequence
 *                    is too short for that (first_frame, length)
 *   stats_host       host, float [3]: mean t_err (per metre), mean r_err (rad per metre), number of segments --
 *                    the two numbers of <seq>-stats.txt.  Synchronises the stream. */
typedef struct davo_kitti_segment {
  int32_t first_frame, last_frame;
  float r_err, t_err, len, speed;       /* as the devkit's `errors` struct (:16-24): errors already divided by len */
} davo_kitti_segment;
int davo_compose_trajectory(davo_ctx*, const float* poses_dev, int n_samples, double* traj_dev, void* cuda_stream);
int davo_kitti_errors(davo_ctx*, const double* gt_dev, const double* res_dev, int n_frames,
                      davo_kitti_segment* seg_dev, float* stats_host, void* cuda_stream);

/* --- real-data input path (SURVEY 8f-2) ---
 * The reference decodes its `<seq>/<id>.jpg` frame triples on the CPU inside tf.data (data_loader.py:241-249,
 * tf.image.decode_jpeg) and feeds uint8 [B,H,3W,3].  davo_decode_jpeg_batch decodes n JPEG byte strings (host memory)
 * with nvJPEG straight into the device tensor davo_forward reads, on `cuda_stream`: image i lands at
 * img_dev + i*H*3W*3, interleaved RGB.  Every image must be H x 3W.  nvJPEG is bound at run time (libnvjpeg.so.12;
 * DAVO_B200_NVJPEG_LIB overrides).  Its pixels are within a few levels of libjpeg's, not identical: the host decode of
 * davo_b200/data_loader.py (PIL) stays the default; this is the throughput option.  Synchronises the stream (nvJPEG's
 * hybrid decoder does its Huffman stage on the host). */
int davo_decode_jpeg_batch(davo_ctx*, const uint8_t* const* jpeg, const int64_t* nbytes, int n, uint8_t* img_dev,
                           void* cuda_stream);

const char* davo_last_error(const davo_ctx*);   /* NULL handle -> last create error */
void davo_destroy(davo_ctx*);
const char* davo_build_info(void);              /* arch / compiler string */
int davo_config_bytes(void);                    /* sizeof(davo_config) in this build: a binding checks its struct against it */

#ifdef __cplusplus
}
#endif
#endif /* DAVO_B200_H */
