/*
 * asm_b200.h -- C ABI of the B200-native (sm_100a) angular-spectrum propagator.
 *
 * The reference (csleemooo/style_transfer_based_holographic_imaging) has no FFI: its boundary for this
 * path is three Python callables,
 *     ASM(O, lamb, d, px, requires_grad=True, zero_padding=False)      utils/Angular_Spectrum_Method.py:7-36
 *     Holo_Generator(args).forward(amplitude, phase, d, ...)           utils/Forward_model.py:16-39
 *     Back_prop(args).forward(holo, d)                                 utils/Forward_model.py:52-65
 * and the backward PyTorch autograd derives from them.  The entry points below are what a ctypes binding of
 * those callables needs (see INTEGRATION.md); each one states the reference lines it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer owned by the caller (PyTorch's
 *     caching allocator), including the workspace.  The library never allocates, frees or retains memory.
 *   - fields are contiguous [B, C, N, N]; N a power of two with 32 <= FFT size <= 4096 (FFT kernels), or any other N
 *     (even when padded) with FFT size <= 2048 (matrix-product path); FFT size = N, or 2N with pad = 1.
 *   - `z` holds one propagation distance in METRES per batch sample (length B; broadcast over C):
 *       z_dtype = ASM_B200_Z_F32: float,  phase constant c = fl32(fl32(2*pi) * z)   (reference with an fp32 tensor d)
 *       z_dtype = ASM_B200_Z_F64: double, phase constant c = 2*pi*z in double        (reference with a python float d)
 *     (utils/Angular_Spectrum_Method.py:29 -- `1j*2*pi*d` is a complex64 product for fp32 d.)
 *   - all work is enqueued asynchronously on `stream` (a cudaStream_t passed as void*); no host sync.
 *   - return value: 0 = ok, negative = ASM_B200_E_* (invalid argument / unsupported shape), positive = cudaError_t.
 *   - thread safe and re-entrant.  The library keeps no caller memory; its only process state is per device and internal:
 *     kernel attributes set once, small sets of internal "lane" streams + fork / join events (the chunks of a call are
 *     issued round-robin on them; up to 4 sets per device, one per caller stream, least recently used set shared beyond
 *     that -- a shared set only adds a false ordering dependency between two caller streams, never a race; host threads
 *     enqueueing on the same set serialise on a mutex while they ENQUEUE, nothing waits for the GPU), and a cache of at
 *     most 8 CUDA graphs per device holding the launch sequences of repeated calls on small transforms (argument values
 *     only; no device memory is retained).  Calls made while the caller's stream is being captured are enqueued plainly.
 */
#ifndef ASM_B200_H_
#define ASM_B200_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ASM_B200_ABI_VERSION 1

/* z_dtype */
#define ASM_B200_Z_F32 0
#define ASM_B200_Z_F64 1

/* in_mode: how (in0, in1) encode the complex input field */
#define ASM_B200_IN_COMPLEX   0 /* in0 = complex64 [B,C,N,N]                          (ASM.py:7, O complex)        */
#define ASM_B200_IN_AMP_PHASE 1 /* in0 = amplitude f32, in1 = phase f32; O = A*exp(i*phase*in_scale)  (Forward_model.py:20-22) */
#define ASM_B200_IN_SQRT_REAL 2 /* in0 = hologram f32 >= 0; O = sqrt(in0)              (Forward_model.py:55)        */
#define ASM_B200_IN_COT_FIELD 3 /* in0 = w f32, in1 = saved field U complex64; O = 2*w*U (cotangent of |U|^2)     */
#define ASM_B200_IN_REAL      4 /* in0 = real f32; O = in0                              (ASM.py:7, O real)           */
#define ASM_B200_IN_CONST_AMP_PHASE 5 /* in0 = ONE f32 amplitude a (device scalar), in1 = phase f32 [B,C,N,N];
                                         O = a*exp(i*phase*in_scale): the loaders' constant amplitude (Data_loader.py:25,:31-32) */

/* out_mode: what is written to (out0, out1) */
#define ASM_B200_OUT_COMPLEX    0 /* out0 = complex64 [B,C,N,N]                         (Forward_model.py:36-37)   */
#define ASM_B200_OUT_INTENSITY  1 /* out0 = |U|^2 f32; if out1 != NULL also out1 = U complex64 (Forward_model.py:39) */
#define ASM_B200_OUT_ABS_ANGLE  2 /* out0 = |U| f32, out1 = angle(U) f32                (Forward_model.py:27-34)   */
#define ASM_B200_OUT_REIM_CAT   3 /* out0 = f32 [B,2,N,N] = cat(re, im) * out_scale, C must be 1 (Forward_model.py:61-65) */
#define ASM_B200_OUT_ABSANG_CAT 4 /* out0 = f32 [B,2,N,N] = cat(|s U|, angle(s U)), s = out_scale (Forward_model.py:58-65) */
#define ASM_B200_OUT_GRAD_AP    5 /* aux0 = amplitude, aux1 = phase; out0 = dL/dA, out1 = dL/dphase (chain rule of :20-22) */

/* Reports ASM_B200_ABI_VERSION of the built library. */
int asm_b200_abi_version(void);

/* Human-readable text for a return code of this library (never NULL). */
const char* asm_b200_strerror(int code);

/* Bytes of device workspace the calls below need for this geometry (tables + L2-resident row/column
 * intermediates for one chunk of samples).  0 if the shape is unsupported. */
size_t asm_b200_workspace_bytes(int B, int C, int N, int pad);

/*
 * Forward propagation  U = crop_N( ifft2( H(z) . fft2( pad(O) ) ) ),  H = exp(i c kz), kz clamped to 0 on
 * evanescent bins.  Replaces ASM (utils/Angular_Spectrum_Method.py:7-36) fused with the input construction of
 * Holo_Generator / Back_prop (Forward_model.py:20-22, :55) and their output stage (:27-39, :56-65).
 *   pad = 0: M = N.   pad = 1: replicate-pad N -> M = 2N, crop back (zero_padding=True, ASM.py:11-14,:34).
 *   in_scale  : phase_normalize (IN_AMP_PHASE), ignored otherwise.
 *   out_scale : amplitude_normalize (OUT_*_CAT), ignored otherwise.
 */
int asm_b200_forward(const void* in0, const void* in1, const void* z, int z_dtype,
                     void* out0, void* out1,
                     int B, int C, int N, int pad, int in_mode, int out_mode,
                     double lambda, double px, float in_scale, float out_scale,
                     void* workspace, size_t workspace_bytes, void* stream);

/*
 * Adjoint propagation (vector-Jacobian product of the forward w.r.t. O, PyTorch convention):
 *   grad_O = replicate_pad^T( ifft2( conj(H) . fft2( zero_embed(g) ) ) )        (SURVEY.md 8a row 6)
 * which is what autograd builds from ASM.py:12,:29-34.  Unpadded it equals ASM(g, -z).
 *   in_mode  : IN_COMPLEX (g) or IN_COT_FIELD (g = 2 w U, backward of |U|^2, Forward_model.py:39).
 *   out_mode : OUT_COMPLEX (grad_O) or OUT_GRAD_AP (aux0 = amplitude, aux1 = phase of the forward call;
 *              out0 = grad_amplitude, out1 = grad_phase; in_scale = phase_normalize).
 */
int asm_b200_adjoint(const void* in0, const void* in1, const void* z, int z_dtype,
                     const void* aux0, const void* aux1, void* out0, void* out1,
                     int B, int C, int N, int pad, int in_mode, int out_mode,
                     double lambda, double px, float in_scale,
                     void* workspace, size_t workspace_bytes, void* stream);

/*
 * Gradient w.r.t. the distance:  grad_z[b] = Re sum_{c,y,x} conj(g) * dU/dz,
 *   dU/dz = crop_N( ifft2( i*K*kz*H . fft2( pad(O) ) ) ),  K = fl32(2*pi) (Z_F32) or 2*pi (Z_F64),
 * i.e. the gradient autograd propagates to `d` because G_in stays in the graph (ASM.py:28-29).
 *   (in0, in1, in_mode, in_scale) describe the forward input O exactly as in asm_b200_forward;
 *   cot_mode = IN_COMPLEX  : cot0 = g complex64
 *   cot_mode = IN_COT_FIELD: cot0 = w f32, cot1 = saved field U complex64 (g = 2 w U)
 *   grad_z: double [B] in metres^-1 units of L; OVERWRITTEN (the call zeroes it first, stream-ordered).
 */
int asm_b200_grad_z(const void* in0, const void* in1, const void* z, int z_dtype,
                    const void* cot0, const void* cot1, int cot_mode, double* grad_z,
                    int B, int C, int N, int pad, int in_mode,
                    double lambda, double px, float in_scale,
                    void* workspace, size_t workspace_bytes, void* stream);

/*
 * 2-D phase unwrapping of B images of H x W wrapped phases (radians, fp32, contiguous), on the device and stream-ordered.
 * Replaces the per-image host loop `unwrap` (utils/functions.py:44-59: .cpu() sync + skimage.restoration.unwrap_phase per
 * image) that Holo_Generator.forward(..., return_field=True, unwrap=True) calls (utils/Forward_model.py:31-32,
 * test_field_retrieval_mnist.py:126).  Same algorithm as scikit-image's 2-D unwrap_phase (Herraez et al. 2002: sort edges by
 * reliability, merge pixel groups along them); ties are broken by edge index instead of skimage's RNG, so results agree
 * wherever the wrapped phase has no residues.  out may alias phase.  Workspace: asm_b200_unwrap_workspace_bytes.
 */
size_t asm_b200_unwrap_workspace_bytes(int B, int H, int W);
int asm_b200_unwrap(const float* phase, float* out, int B, int H, int W,
                    void* workspace, size_t workspace_bytes, void* stream);

/*
 * Focal stack: every sample propagated to K distances.  Plane (b, k) equals asm_b200_forward of sample b at distance
 * z[b*K + k] with C = 1.  The forward row FFT of a sample runs once and is shared by its K planes (its spectrum stays in
 * the L2-resident workspace); each plane then costs the column pass and the inverse row pass.
 *   z        : [B][K] distances in metres, z_dtype as in the Conventions (Z_F32: c = fl32(fl32(2 pi) z); Z_F64: 2 pi z).
 *   in_mode  : IN_COMPLEX, IN_REAL, IN_SQRT_REAL (hologram -> sqrt on load, as Back_prop), IN_AMP_PHASE or
 *              IN_CONST_AMP_PHASE, with in0 / in1 / in_scale as in asm_b200_forward for C = 1.
 *   out_mode : OUT_COMPLEX, OUT_INTENSITY or OUT_ABS_ANGLE; out0 (and out1 = angle planes, OUT_ABS_ANGLE only; NULL
 *              otherwise) are [B][K][N][N].  out0 = NULL: no image output at all (moments only).
 *   moments  : double [B][K][3] = (Sum |U|, Sum |U|^2, Sum |U|^4) over the N x N output window; overwritten.  NULL: none.
 *              Reduced from per-row partials in a fixed order (no atomics): repeated calls are bit-identical.
 * Returns E_NULL if out0 and moments are both NULL; E_SHAPE for B <= 0, K <= 0 or an N / pad that
 * asm_b200_workspace_bytes rejects; E_MODE for another in/out mode or a non-NULL out1 outside OUT_ABS_ANGLE; otherwise
 * the codes of the other calls.  Like every call here: stream-ordered on `stream`, no host sync, nothing retained.
 * asm_b200_focal_stack_workspace_bytes: the workspace it needs (0 = unsupported); never less than
 * asm_b200_workspace_bytes(B, 1, N, pad), so the same buffer also serves asm_b200_forward of the samples.
 */
size_t asm_b200_focal_stack_workspace_bytes(int B, int K, int N, int pad);
int asm_b200_focal_stack(const void* in0, const void* in1, const void* z, int z_dtype, int K,
                         void* out0, void* out1, double* moments,
                         int B, int N, int pad, int in_mode, int out_mode,
                         double lambda, double px, float in_scale,
                         void* workspace, size_t workspace_bytes, void* stream);

/* Number of CUDA kernels this library has launched in this process so far (all threads, all devices).
 * Instrumentation for bench.py (`gpu_launches`); not part of the reference's interface. */
unsigned long long asm_b200_launch_count(void);

/* Instrumentation: ms3 (may be NULL) receives the accumulated device time in ms of the three passes
 * {row FFT, column FFT.H.IFFT, row IFFT} recorded with CUDA events since profiling was enabled; then
 * enable = 1/0 switches per-pass timing on/off and clears the accumulators (enable < 0: leave unchanged).
 * Profiling mode synchronises after every chunk -- never leave it on while measuring throughput. */
void asm_b200_profile(int enable, double* ms3);

/* error codes (negative return values) */
#define ASM_B200_E_NULL        (-1) /* a required pointer is NULL                      */
#define ASM_B200_E_SHAPE       (-2) /* unsupported N (see Conventions) / B,C <= 0        */
#define ASM_B200_E_MODE        (-3) /* unknown or inconsistent in_mode / out_mode      */
#define ASM_B200_E_WORKSPACE   (-4) /* workspace too small or misaligned (256 B)       */
#define ASM_B200_E_OPTICS      (-5) /* lambda or px not finite and positive            */
#define ASM_B200_E_DRIVER      (-6) /* cuTensorMapEncodeTiled unavailable / failed     */
#define ASM_B200_E_DEVICE      (-7) /* current device is not compute capability 10.x   */

#ifdef __cplusplus
}
#endif
#endif /* ASM_B200_H_ */
