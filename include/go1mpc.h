/*
 * go1mpc.h -- C ABI of libgo1mpc.so: batched, B200-native (sm_100a, FP64)
 * implementation of the Go1 gait-planning MPC hot path of
 * jtdingx/quadrupedal_loco.  Plain pointers and sizes only; no C++ or torch
 * types cross this boundary.  Every entry point returns 0 on success or a
 * negative GO1MPC_E_* code; go1mpc_last_error() gives the text.  There is no
 * CPU fallback: without a CUDA device every compute call fails.
 *
 * Reference abbreviations (paths under the reference repository):
 *   RT  = unitree_ros/rt_mpc_qp/src        NLP = unitree_ros/mosek_nlp_kmp/src
 *   GO1 = unitree_ros/go1_rt_control/src
 *
 * The reference has no FFI: its seams are C++ classes.  Each function below
 * names the class method(s) it replaces; the C++ mirror of those classes that
 * binds to this ABI is in quadrupedal_loco_b200/host/ and INTEGRATION.md shows
 * the binding a maintainer of the reference would add.
 *
 * QP convention (RT/utils/EiQuadProg/EiQuadProg.hpp:15-32):
 *     min 0.5 x'Gx + g0'x   s.t.  CE'x + ce0 = 0,  CI'x + ci0 >= 0
 * Matrices are column-major double, one constraint per column of CE / CI.
 *
 * Batch layout ("field arrays of per-problem blocks"): every argument is one
 * array per field; problem b owns the contiguous block [b*stride, (b+1)*stride).
 * A warp (or thread) works on one problem, so a block is read with fully
 * coalesced 128-byte lines or one TMA bulk copy; blocks that are TMA sources
 * are documented as 16-byte aligned with an even number of doubles.
 * Pointers suffixed _d are DEVICE pointers owned by the caller; the *_host
 * variants take HOST pointers and do the staging copies inside the call.
 * `stream` is a cudaStream_t passed as void* (NULL = the handle's own stream).
 * A handle is thread-compatible, not thread-safe; use one per host thread/GPU.
 */
#ifndef GO1MPC_H
#define GO1MPC_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GO1MPC_VERSION_STRING "0.1.0"
#define GO1MPC_FOOTSTEPS 27          /* _footstepsnumber, RT/FastMPC/PRMPCClass.h:30 */
#define GO1MPC_BODY_NH_MAX 40

/* error codes (function return values) */
enum {
    GO1MPC_OK = 0,
    GO1MPC_E_INVALID = -1,     /* bad argument (size, NULL, alignment)        */
    GO1MPC_E_CUDA = -2,        /* CUDA runtime error, see go1mpc_last_error   */
    GO1MPC_E_NO_DEVICE = -3,   /* no usable CUDA device: there is no fallback */
    GO1MPC_E_UNSUPPORTED = -4  /* size outside what the kernels are built for */
};

/* per-problem solver status (status_d[b]); numerically = oracle's ORC_* */
enum {
    GO1MPC_QP_OK = 0,            /* converged                                  */
    GO1MPC_QP_NOT_PD = 1,        /* LLT failed: x untouched, cost = +inf       */
    GO1MPC_QP_INFEASIBLE = 2,    /* no step possible: cost = +inf              */
    GO1MPC_QP_ITER_CAP = 3,      /* safety cap hit (reference has no cap)      */
    GO1MPC_QP_NAN = 4,           /* NaN in x  (reference: solveQP() == false)  */
    GO1MPC_QP_EQ_DEPENDENT = 5,  /* dependent equalities: early return         */
    GO1MPC_QP_SKIPPED = -1       /* front-end gated this tick: no solve ran    */
};
/* iters_d[b*GO1MPC_ITERS + k]: outer passes (step 1), constraints added, dropped,
 * degenerate restarts, passes through step 2a, and the ALGORITHMIC flop count of the
 * dense reference algorithm along the path this problem took (SURVEY.md section 8d:
 * what the roofline figure uses; saturates at INT_MAX). */
#define GO1MPC_ITERS 6
enum { GO1MPC_IT_OUTER = 0, GO1MPC_IT_ADD = 1, GO1MPC_IT_DROP = 2, GO1MPC_IT_DEGEN = 3,
       GO1MPC_IT_L2A = 4, GO1MPC_IT_FLOPS = 5 };

/* Constants of the body-inclination MPC.  Defaults = the reference's
 * compile-time values: RT/Robotpara/robot_const_para_config.cpp:8-47,
 * RT/FastMPC/PRMPCClass.cpp:157-170,227-261,280-287. */
typedef struct {
    double dt_mpc;               /* 0.01   gait::dt_mpc_fast                   */
    double dt_slow;              /* 0.025  gait::dt_mpc_slow                   */
    double tstep;                /* 0.7    gait::t_period                      */
    double height_offset_time;   /* 1.0                                        */
    double g, mass, j_ini;       /* 9.8, 12, 12*0.1*0.1                        */
    double foot_length, foot_width; /* 0.02, 0.02                              */
    double theta_lim;            /* 10 deg in rad                              */
    double torque_lim;           /* 20 (the reference divides it by j_ini)     */
    double Rtheta, alphatheta, beltatheta, gama_zmp; /* 100, 10, 5e9, 5000     */
    double lamda[4];             /* state feedback gains (all 0 as shipped)    */
} Go1BodyMpcConfig;

/* Constants of the step-location / step-timing SQP.  Defaults = the reference's values:
 * NLP/NLP/NLPClass_sqp.cpp:212-214,244-258,273-286 (go1 weights), NLP/NLP/NLPClass.h:30-38,
 * NLP/NLPRTControl/NLPRTControlClass.cpp:35-42. */
typedef struct {
    double dt;                   /* 0.025  _dt                                  */
    double Wn;                   /* sqrt(g / hcom), hcom = 0.309458             */
    double ggg;                  /* 9.8                                         */
    double t_min, t_max;         /* 0.5, 1.0  step-period bounds                */
    double footx_max, footx_min; /* 0.15, -0.05                                 */
    double footx_vmax, footx_vmin, footy_vmax, footy_vmin;  /* 3, -2.875, 2, -1 */
    double comax_max, comax_min, comay_max, comay_min;      /* 5, -5, 6, -6     */
    double aax, aay, aaxv, aayv, bbx, bby, rr1, rr2;        /* 5e4 5e4 1e3 5e2 2e6 1e7 1e6 1e6 */
    double half_hip_width, foot_width;                       /* 0.12675, 0.03    */
    double lamda[4];             /* com x, vx, y, vy feedback gains (0 as shipped) */
    double hcom;                 /* 0.309458  RobotPara_Z_C - _height_offset    */
    int ext_height;              /* 0: CoM_height_solve on the device; 1: comz/comaz/comvz from in_d */
    int reserved;
    double stepwidth0;           /* 0.12675  _stepwidth(0) = stepwidthinput / 2 (NLPClass_sqp.cpp:66-67) */
    double lift_height;          /* 0.03     _lift_height (NLPRTControlClass.cpp:48), 0 for the last two steps */
} Go1StepMpcConfig;

typedef struct {
    Go1BodyMpcConfig body;
    Go1StepMpcConfig step;
    int qp_iter_cap_scale;       /* cap on step-2a passes = scale*(n+m+p)+50; default 20 */
    int reserved[7];
} Go1MpcConfig;

typedef struct go1mpc go1mpc_t;

const char *go1mpc_version(void);
int go1mpc_config_default(Go1MpcConfig *cfg);
/* device < 0 selects the current CUDA device */
int go1mpc_create(const Go1MpcConfig *cfg, int device, go1mpc_t **out);
void go1mpc_destroy(go1mpc_t *h);
const char *go1mpc_last_error(const go1mpc_t *h);
int go1mpc_device(const go1mpc_t *h);
/* number of kernels this handle has launched so far (bench's gpu_launches) */
long long go1mpc_launch_count(const go1mpc_t *h);
/* the handle's own cudaStream_t (as void*), e.g. to record timing events on it */
void *go1mpc_stream(const go1mpc_t *h);
/* multiprocessor count of the handle's device */
int go1mpc_sm_count(const go1mpc_t *h);
/* device-to-device copy on `stream` (NULL = the handle's): all per-instance state of this library
 * is plain SoA / record memory, so checkpointing or restoring a batch is a memcpy */
int go1mpc_copy_device_async(go1mpc_t *h, void *dst_d, const void *src_d, size_t bytes, void *stream);
/* The *_host_async entries order calls that share a device-resident buffer (planner state, body records) through a per-buffer
 * event; call this before freeing such a buffer (waits for its last user, drops the bookkeeping). */
int go1mpc_forget_buffer(go1mpc_t *h, const void *buf_d);
/* wait for the handle's stream and for every pipelined *_host_async call */
int go1mpc_synchronize(go1mpc_t *h);

/* ---------------------------------------------------------------------------
 * Generic dense QP batch.  Replaces, for B independent problems of one shape,
 *   QPBaseClass::solveQP            RT/QP/QPBaseClass.cpp:126-153
 *   Eigen::QP::solve_quadprog       RT/utils/EiQuadProg/EiQuadProg.cpp:493-513
 * Strides (doubles): G n*n, g0 n, CE n*p, ce0 p, CI n*m, ci0 m, x n, cost 1;
 * (ints): active m+p, nactive 1, iters GO1MPC_ITERS, status 1.  CE_d/ce0_d may be NULL
 * when p == 0.  x_d is in/out (left untouched when G is not PD, as the
 * reference does).  active_d/nactive_d/iters_d/cost_d may be NULL.
 * Limits: n <= 96, m + p <= 1024.
 * ------------------------------------------------------------------------ */
int go1mpc_qp_solve_batch(go1mpc_t *h, int n, int p, int m, int B,
                          const double *G_d, const double *g0_d,
                          const double *CE_d, const double *ce0_d,
                          const double *CI_d, const double *ci0_d,
                          double *x_d, double *cost_d,
                          int *active_d, int *nactive_d, int *iters_d, int *status_d,
                          void *stream);
int go1mpc_qp_solve_batch_host(go1mpc_t *h, int n, int p, int m, int B,
                               const double *G, const double *g0,
                               const double *CE, const double *ce0,
                               const double *CI, const double *ci0,
                               double *x, double *cost,
                               int *active, int *nactive, int *iters, int *status);

/* ---------------------------------------------------------------------------
 * Body-inclination MPC tick for B independent instances, horizon nh.
 * Replaces PRMPCClass::body_theta_mpc (condensation + QP + clamp + roll-out)
 *   RT/FastMPC/PRMPCClass.cpp:379-714, solve_body_rotation/Solve :799-849,
 *   Indexfind :716-738, with the model of Initialize :198-261,280-287.
 * One launch: condensation, the 2nh-variable / 12nh-row QP and the
 * post-processing are fused; the QP matrices never exist in HBM.
 *
 * in_d   [B][go1mpc_body_in_stride(nh)] doubles, 16-byte aligned, per problem:
 *          [0,27)      tx        step-cycle start times (_tx)
 *          [27]        tick      i, stored as a double (exact integer)
 *          [28,32)     theta     (thetaxk0, thetaxk1, thetayk0, thetayk1)
 *          [32,36)     bodyangle_state (only used with non-zero lamda)
 *          [36,36+2nh) x_warm    _V_ini (kept when G is not PD / tick gated)
 *          then 9 rows of nh:  zmp_x, zmp_y, ang_x, ang_y, rfoot_x, rfoot_y,
 *                              lfoot_x, lfoot_y, comacc_z
 *          (+1 pad double when the count is odd)
 * out_d  [B][go1mpc_body_out_stride(nh)] doubles, in/out (a gated tick keeps
 *        its out14, as the reference returns its stale members):
 *          [0,14)      out14     = the Vec14 body_theta_mpc returns (:696-709)
 *          [14,18)     theta     updated state
 *          [18,18+2nh) x         _V_ini after the tick
 *          [18+2nh]    cost
 *          (+pad to an even count)
 * diag_d [B][go1mpc_body_diag_stride(nh)] ints (may be NULL):
 *          [0] status  [1] nactive  [2,6) iters  [6] bjx1  [7] bjx2
 *          [8] passes through step 2a  [9] algorithmic flops (GO1MPC_IT_FLOPS)
 *          [10, 10+2nh) final active set (constraint indices, Appendix E of SURVEY.md)
 * Supported nh: 3..40 (the reference compiles nh = 4).
 * ------------------------------------------------------------------------ */
int go1mpc_body_in_stride(int nh);
int go1mpc_body_out_stride(int nh);
int go1mpc_body_diag_stride(int nh);
int go1mpc_body_mpc_step_batch(go1mpc_t *h, int nh, int B,
                               const double *in_d, double *out_d, int *diag_d,
                               void *stream);
/* Diagnostic: number of instances the roll/pitch-split kernel handed to the combined-solve kernel
 * (infeasible / degenerate / non-converged halves) since the handle was created.  Synchronises the device. */
int go1mpc_body_handover_total(go1mpc_t *h, long long *total);
/* Diagnostic: warps of the body solve kernel that left through its defensive iteration guard (0 unless
 * there is a bug).  Synchronises the device. */
int go1mpc_body_guard_trips(go1mpc_t *h, long long *total);
int go1mpc_body_mpc_step_batch_host(go1mpc_t *h, int nh, int B,
                                    const double *in, double *out, int *diag);
/* Pipelined host entries: enqueue H2D copy, kernel and D2H copy on one of the handle's eight
 * internal lanes (consecutive calls use consecutive lanes, so the copies of one batch overlap
 * the kernels of its neighbours) and return at once; go1mpc_synchronize() waits for all of
 * them.  Host buffers should be pinned and must stay untouched until then.  The planner state
 * of the step-timing tick stays RESIDENT ON THE DEVICE (state_d / state_out_d are device
 * pointers, as in go1mpc_step_timing_step_batch); only the per-tick inputs and results move.
 * Calls that write a state buffer an earlier pipelined call wrote are ordered after it. */
int go1mpc_body_mpc_step_batch_host_async(go1mpc_t *h, int nh, int B,
                                          const double *in, double *out, int *diag);
int go1mpc_step_timing_step_batch_host_async(go1mpc_t *h, int n_sqp, int B, const int *tick,
                                             const double *state_d, double *state_out_d,
                                             const double *in, double *out, int *diag);
/* Pipelined body tick with the slow part of the record RESIDENT ON THE DEVICE, as the planner state is:
 * what PRMPCClass::body_theta_mpc takes per call (RT/FastMPC/PRMPCClass.cpp:379-395) moves, what the class
 * keeps as members (_tx :174-178, _V_ini :258-261, the stale results a gated tick returns) stays in HBM.
 *   tx_d     device [B][28] doubles: tx[27] + 1 pad (the caller rewrites a row when the planner re-times a step)
 *   out_d    device [B][go1mpc_body_out_stride(nh)], in/out: the output records of go1mpc_body_mpc_step_batch;
 *            the tick reads its warm start x (and, when gated, its out14) from here and writes its results back
 *   tick_in  host [B][go1mpc_body_tick_in_stride(nh)]: tick | theta(4) | bodyangle_state(4) | 9 rows of nh
 *            (= record doubles [27,36) and [36+2nh, 36+11nh) of the full format; + pad to an even count)
 *   tick_out host [B][GO1MPC_BODY_TICK_OUT]: out14 | theta(4) | cost | 0
 *   diag     host [B][go1mpc_body_diag_stride(nh)] or NULL
 * Results are bit-identical to the full-record entries.  Calls on the same out_d are ordered. */
#define GO1MPC_BODY_TICK_OUT 20
int go1mpc_body_tick_in_stride(int nh);
int go1mpc_body_mpc_step_batch_resident_host_async(go1mpc_t *h, int nh, int B,
                                                   const double *tx_d, double *out_d,
                                                   const double *tick_in, double *tick_out, int *diag);

/* Model matrices the handle condenses with, for inspection/tests (host
 * buffers, column-major): pps,pvs nh x 2; ppu,pvu,ppu_2,pvu_2 nh x nh.
 * Replaces PRMPCClass::Matrix_ps / Matrix_pu, RT/FastMPC/PRMPCClass.cpp:741-796. */
int go1mpc_body_model(go1mpc_t *h, int nh, double *pps, double *pvs,
                      double *ppu, double *pvu, double *ppu_2, double *pvu_2);
/* default step table _tx of PRMPCClass::Initialize (:174-178), 27 doubles */
int go1mpc_body_default_tx(go1mpc_t *h, double *tx27);

/* ---------------------------------------------------------------------------
 * Step-location / step-timing SQP tick (40 Hz planner) for B independent instances.
 * Replaces NLPClass::step_timing_opti_loop  NLP/NLP/NLPClass_sqp.cpp:693-1102 with
 *   step_timing_object_function :1144-1173, step_timing_constraints :1175-1458,
 *   solve_stepping_timing/Solve :1613-1653 (QP n=4, p=1, m=24), Indexfind :1105-1141.
 * One launch runs n_sqp SQP iterations (reference: 3; 1..5 supported), the write-back of
 * step length / width / period and of the step tables, the LIPM roll-out of samples
 * i..i+2, the feedback blend, the integer step indices and CoM_height_solve (:2361-2473,
 * the 6th-order vertical CoM polynomial).
 *
 * Layout: STRUCTURE OF ARRAYS, element-major / batch-minor: field f of instance b is
 * at [f*B + b] (one thread per instance: every access of a warp is coalesced).
 * tick_d  [B] ints         i of the reference (>= 1); an instance with tick < 1 is skipped (nothing read or written)
 * state_d [202][B] doubles, the planner state before the tick; state_out_d receives the
 *         state after it and may be the same buffer (in-place: only changed fields are
 *         written).  Fields:
 *           [0,27) ts   [27,54) tx   [54,81) footx_ref  [81,108) footy_ref
 *           [108,135) footz_ref  [135,162) Lxx_ref  [162,189) Lyy_ref
 *           [189,195) com x,vx,ax,y,vy,ay _feed at tick i-1
 *           [195,199) _Vari_ini.col(i-1) = (Lx, Ly, cosh(w T), sinh(w T))
 *           [199,201) _comvx_endref, _comvy_endref   [201] _bjx1 of the previous tick (exact integer)
 * in_d    [20][B] doubles: [0,6) estimated com x,vx,ax,y,vy,ay  [6,8) right foot x,y
 *           [8,10) left foot x,y  [16,19) Zsc(i..i+2) (terrain height under the CoM)
 *           [10,13) comz(i..i+2)  [13,16) comaz  [19] comvz(i): read only when cfg.step.ext_height != 0
 * out_d   [38][B] doubles = the Vec38 the reference returns (:1048-1090)
 * diag_d  [60][B] ints (may be NULL): [0] period index (_periond_i; -1 = time beyond the
 *           step table, nothing written)  [1] k_yu  [2] bjxx  [3] bjx1  [4] QPs solved;
 *           then per SQP iteration q < 5, at 5 + 11 q: status (-1 = no solve), nactive,
 *           iters[4], active set[5] (slot 0 = -1 is the equality)
 * ------------------------------------------------------------------------ */
#define GO1MPC_STEP_STATE_DOUBLES 202
#define GO1MPC_STEP_IN_DOUBLES 20
#define GO1MPC_STEP_OUT_DOUBLES 38
#define GO1MPC_STEP_DIAG_INTS 60
int go1mpc_step_timing_step_batch(go1mpc_t *h, int n_sqp, int B, const int *tick_d,
                                  const double *state_d, double *state_out_d,
                                  const double *in_d, double *out_d,
                                  int *diag_d, void *stream);
int go1mpc_step_timing_step_batch_host(go1mpc_t *h, int n_sqp, int B, const int *tick,
                                       double *state, const double *in, double *out, int *diag);
/* Initial step tables of one planner (host buffer, 202 doubles, instance-major):
 * NLPClass::FootStepInputs :51-75 and Initialize :131-206 for the given step length,
 * width and height (reference: 0.075, 0.2535, 0) and period tstep (0.7). */
int go1mpc_step_default_state(go1mpc_t *h, double steplength, double stepwidth,
                              double stepheight, double tstep, double *state201);

/* ---------------------------------------------------------------------------
 * Go1 leg kinematics for B independent legs.  Replaces Kinematicclass
 * (GO1/kinematics/Kinematics.h:49-60, Kinematics.cpp:29-304):
 *   go1mpc_leg_fk_batch  -> Forward_kinematics (body_p_d == NULL) / Forward_kinematics_g
 *   go1mpc_leg_ik_batch  -> Inverse_kinematics (body_p_d == NULL: <= 10 updates, stop
 *                           max(dq) < 1e-4 without abs, as the reference) / Inverse_kinematics_g
 *                           (<= 15 updates, stop |dp|^2 <= 1e-6); lamda = 0.5
 * The reference returns the Jacobian through the member Jacobian_kin read after each
 * call (servo.cpp:734-741,1038-1051); here it is the output array jac_d.
 * Layout: structure of arrays, [f*B + b].  q_d / qini_d / pdes_d / pos_d / body_p_d /
 * body_r_d (roll, pitch, yaw): [3][B] doubles; jac_d: [9][B] doubles, row-major 3x3, may be
 * NULL; leg_d: [B] ints, 0 FR, 1 FL, 2 RR, 3 RL; iters_d: [B] ints (Newton updates), may be NULL.
 * ------------------------------------------------------------------------ */
int go1mpc_leg_fk_batch(go1mpc_t *h, int B, const double *q_d, const int *leg_d,
                        const double *body_p_d, const double *body_r_d,
                        double *pos_d, double *jac_d, void *stream);
int go1mpc_leg_ik_batch(go1mpc_t *h, int B, const double *pdes_d, const double *qini_d, const int *leg_d,
                        const double *body_p_d, const double *body_r_d,
                        double *q_d, double *jac_d, int *iters_d, void *stream);
int go1mpc_leg_fk_batch_host(go1mpc_t *h, int B, const double *q, const int *leg,
                             const double *body_p, const double *body_r, double *pos, double *jac);
int go1mpc_leg_ik_batch_host(go1mpc_t *h, int B, const double *pdes, const double *qini, const int *leg,
                             const double *body_p, const double *body_r, double *q, double *jac, int *iters);

/* ---------------------------------------------------------------------------
 * Swing-foot trajectory of the step planner for B instances; run after the step-timing tick
 * of the same index.  Replaces NLPClass::Foot_trajectory_solve_mod2 (NLP/NLP/NLPClass_sqp.cpp:
 * 2039-2358) and solve_AAA_inv2 (:3633-3645); the stop-walking branch is go1mpc_foot_trajectory_stop_batch.
 * SoA layout [f*B + b].  Instances with tick < 1 are skipped.
 * state_d [202][B]  planner state AFTER go1mpc_step_timing_step_batch;  out38_d [38][B] its output
 * foot_d  [32][B] in/out, the window of the reference's whole-walk foot arrays:
 *           [0,6) R xyz, L xyz at tick j-1   [6,12) what the arrays hold at j   [12,18) at j-2
 *           [18,24) at j-3   [24,30) frozen at the step's start   [30] step start index the freeze
 *           belongs to (-1 none)   [31] _ry_left_right.  Initial value: go1mpc_foot_default_state.
 * out18_d [18][B] = the Vec18 of the reference (R xyz, L xyz | velocities | accelerations)
 * right_support_d [B] ints (0 left support, 1 right support, 2 double support), may be NULL
 * ------------------------------------------------------------------------ */
#define GO1MPC_FOOT_STATE_DOUBLES 32
#define GO1MPC_FOOT_OUT_DOUBLES 18
int go1mpc_foot_trajectory_batch(go1mpc_t *h, int B, const int *tick_d, const double *state_d,
                                 const double *out38_d, double *foot_d, double *out18_d,
                                 int *right_support_d, void *stream);
int go1mpc_foot_trajectory_batch_host(go1mpc_t *h, int B, const int *tick, const double *state,
                                      const double *out38, double *foot, double *out18, int *right_support);
int go1mpc_foot_default_state(go1mpc_t *h, double *foot32);
/* The same with the stop-walking branch (:2043-2048): lift0_d [B] doubles, in/out -- the first step index whose lift height is
 * zeroed (initially GO1MPC_FOOTSTEPS = none); stop_d [B] doubles or NULL -- the caller's _stopwalking flag (non-zero = set).
 * A tick beyond _t_end_footstep (go1mpc_nlp_t_end_footstep) acts like a stop, as in the reference. */
int go1mpc_foot_trajectory_stop_batch(go1mpc_t *h, int B, const int *tick_d, const double *state_d, const double *out38_d,
                                      double *foot_d, double *out18_d, int *right_support_d, double *lift0_d,
                                      const double *stop_d, void *stream);
int go1mpc_foot_trajectory_stop_batch_host(go1mpc_t *h, int B, const int *tick, const double *state, const double *out38,
                                           double *foot, double *out18, int *right_support, double *lift0, const double *stop);

/* ---------------------------------------------------------------------------
 * Servo kinematics tick for B robots (cfg5's fused leg IK / Jacobian stage).  Replaces the
 * leg mapping and the four Inverse_kinematics_g calls of go1_servo's 1 kHz loop,
 * GO1/servo_control/servo.cpp:935-1051: foot target of each leg = its homing position + the
 * planner's virtual right / left foot displacement -+ half hip width, the virtual foot chosen
 * by gait_mode (101 pace, 102 trot, 103 gallop; servo.h:100-102), body pose = (com x, com y *
 * y_offset, com z; roll, pitch, yaw), initial guess = the previous joint angles.
 * SoA [f*B + b]: com_d, theta_d, rfoot_d, lfoot_d [3][B]; homing_d [12][B] and q_d [12][B]
 * (in/out) leg-major in the order FR, FL, RR, RL; jac_d [36][B] (row-major 3x3 per leg),
 * foot_des_d [12][B], iters_d [4][B] may be NULL.
 * ------------------------------------------------------------------------ */
int go1mpc_servo_kin_tick_batch(go1mpc_t *h, int B, int gait_mode, double y_offset,
                                const double *com_d, const double *theta_d,
                                const double *rfoot_d, const double *lfoot_d, const double *homing_d,
                                double *q_d, double *jac_d, double *foot_des_d, int *iters_d, void *stream);

/* ---------------------------------------------------------------------------
 * Fused control tick for B robots (SURVEY.md 8b / cfg5): ONE call enqueues, on one stream and with every
 * intermediate resident on the device,
 *   1. the step-location / step-timing SQP tick   (= go1mpc_step_timing_step_batch, state updated in place)
 *   2. the planner's swing-foot trajectory        (= go1mpc_foot_trajectory_batch on the new state / out38)
 *   3. the body-inclination MPC tick               (= go1mpc_body_mpc_step_batch)
 *   4. the servo kinematics tick                   (= go1mpc_servo_kin_tick_batch) with the body pose taken from the
 *      ticks above: position = planner CoM (out38 rows 0..2), roll / pitch = body-MPC angles (out record [0], [1]),
 *      yaw 0; virtual right / left foot = swing-foot positions (out18 rows 0..2 / 3..5)
 *   5. optionally the GRF QP and the torque map    (= go1mpc_grf_force_opt_batch, go1mpc_grf_joint_torques_batch on stage 4's
 *      Jacobians and the QP's forces: Dynamiccclass::force_opt / compute_joint_torques, servo.cpp:1200-1243)
 * i.e. NLPClass::step_timing_opti_loop + Foot_trajectory_solve_mod2 -> PRMPCClass::body_theta_mpc -> the leg mapping
 * and four Inverse_kinematics_g of GO1/servo_control/servo.cpp:935-1051 without a host round trip.  Results are
 * bit-identical to calling the four entry points in that order.  All pointers are device pointers with the layouts
 * of the individual entry points; servo_theta_d [3][B] is scratch the call fills (roll, pitch, yaw).
 * ------------------------------------------------------------------------ */
typedef struct {
  int n_sqp;                    /* 1: planner */
  const int *tick_d;
  double *step_state_d;         /*    [202][B], in place */
  const double *step_in_d;      /*    [20][B] */
  double *out38_d;              /*    [38][B] */
  int *step_diag_d;             /*    [60][B] or NULL */
  double *foot_d;               /* 2: [32][B] in/out */
  double *out18_d;              /*    [18][B] */
  int *right_support_d;         /*    [B] or NULL */
  int nh;                       /* 3: body MPC */
  const double *body_in_d;      /*    [B][go1mpc_body_in_stride(nh)] */
  double *body_out_d;           /*    [B][go1mpc_body_out_stride(nh)] in/out */
  int *body_diag_d;             /*    [B][go1mpc_body_diag_stride(nh)] or NULL */
  int gait_mode;                /* 4: servo kinematics (101 pace, 102 trot, 103 gallop) */
  double y_offset;
  const double *homing_d;       /*    [12][B] */
  double *q_d;                  /*    [12][B] in/out */
  double *jac_d;                /*    [36][B] or NULL */
  double *foot_des_d;           /*    [12][B] or NULL */
  int *ik_iters_d;              /*    [4][B] or NULL */
  double *servo_theta_d;        /*    [3][B] scratch (filled by the call) */
  const double *grf_in_d;       /* 5: optional (NULL skips it): force QP records [B][48] of go1mpc_grf_force_opt_batch */
  double *grf_out_d;            /*    [B][16] */
  int *grf_diag_d;              /*    [B][32] or NULL */
  const int *swing_d;           /*    torque map (tau_d NULL skips it): [4][B] */
  const double *p_des_d, *p_est_d, *pv_des_d, *pv_est_d;   /* [12][B] each */
  double *tau_d;                /*    [12][B]: -J' f + gravity term from stage 4's jac_d and the QP's forces */
} Go1FusedTick;
int go1mpc_fused_tick_batch(go1mpc_t *h, int B, const Go1FusedTick *t, void *stream);

/* ---------------------------------------------------------------------------
 * Ground-reaction-force distribution of go1_servo's 1 kHz loop for B robots.  Replaces
 * Dynamiccclass (GO1/whole_body_dynamics/dynmics_compute.cpp):
 *   go1mpc_grf_force_distribution_batch -> force_distribution :141-261 (gait_mode 101 / 102)
 *   go1mpc_grf_force_opt_batch          -> force_opt :265-373 + solve_grf_opt :387-427: the
 *       12-variable QP (alpha 1e4, beta 1e3, gama 10, fz_max 160, mu 0.25 of :55-66) with 12
 *       equality columns (identity on the legs that must carry no force, all-zero -- and
 *       skipped by the solver -- on the others) and 24 inequalities; on a NaN solution the
 *       closed-form guess is returned, as the reference does.
 * force_opt records are instance-major:
 *   in_d  [B][48]: base_p 3 | leg_p 12 (FR, FL, RR, RL xyz) | FT_total_des 6 | F_leg_guess 12 |
 *                  previous grf_opt 12 | gait_mode | right_support | pad
 *   out_d [B][16]: grf_opt 12 | cost | qp_solution (1/0) | pad 2
 *   diag_d [B][32] ints (may be NULL): status, nactive, iters[4], qp_solution, 0, active set[24]
 * force_distribution is SoA [f*B + b]: com_des [3][B], leg_des [12][B], F_force_des [6][B]
 * (L xyz, R xyz), rfoot_des / lfoot_des [3][B] -> F_leg_ref [12][B] (= F_leg_guess).
 * ------------------------------------------------------------------------ */
int go1mpc_grf_force_opt_batch(go1mpc_t *h, int B, const double *in_d, double *out_d, int *diag_d, void *stream);
int go1mpc_grf_force_distribution_batch(go1mpc_t *h, int B, int gait_mode, double y_coefficient,
                                        const double *com_des_d, const double *leg_des_d, const double *F_force_des_d,
                                        const double *rfoot_des_d, const double *lfoot_des_d,
                                        double *F_leg_ref_d, void *stream);
/* Joint torques of the four legs.  Replaces Dynamiccclass::compute_joint_torques :109-138 as go1_servo calls it once per
 * leg (GO1/servo_control/servo.cpp:1232-1243, leg_number 0..3 = FR, FL, RR, RL):
 *   tau = -Jaco' * w + gravity_compensate(:, leg),   w = swing_kp (p_des - p_est) + swing_kd (pv_des - pv_est) for a
 *   swing leg (swing_kp 1, swing_kd 0.01, :37-38), the leg's column of F_leg_ref for a stance leg.
 * SoA [f*B + b]: jac_d [36][B] (row-major 3x3 per leg, the layout go1mpc_servo_kin_tick_batch / go1mpc_leg_ik_batch
 * write), swing_d [4][B] ints, p_des_d / p_est_d / pv_des_d / pv_est_d [12][B], tau_d [12][B].  F_leg_ref element k of
 * robot b is read at F_leg_ref_d[k * F_elem_stride + b * F_robot_stride]: (B, 1) for the SoA output of
 * go1mpc_grf_force_distribution_batch, (1, 16) for the out records of go1mpc_grf_force_opt_batch. */
int go1mpc_grf_joint_torques_batch(go1mpc_t *h, int B, const double *jac_d, const int *swing_d,
                                   const double *p_des_d, const double *p_est_d,
                                   const double *pv_des_d, const double *pv_est_d,
                                   const double *F_leg_ref_d, long long F_elem_stride, long long F_robot_stride,
                                   double *tau_d, void *stream);

/* Synchronous host-buffer forms of the three entries above (same layouts, host pointers; what the C++ mirror of
 * Dynamiccclass in host/go1mpc.hpp calls with B = 1). */
int go1mpc_grf_force_opt_batch_host(go1mpc_t *h, int B, const double *in, double *out, int *diag);
int go1mpc_grf_force_distribution_batch_host(go1mpc_t *h, int B, int gait_mode, double y_coefficient,
                                             const double *com_des, const double *leg_des, const double *F_force_des,
                                             const double *rfoot_des, const double *lfoot_des, double *F_leg_ref);
int go1mpc_grf_joint_torques_batch_host(go1mpc_t *h, int B, const double *jac, const int *swing,
                                        const double *p_des, const double *p_est,
                                        const double *pv_des, const double *pv_est,
                                        const double *F_leg_ref, long long F_elem_stride, long long F_robot_stride,
                                        double *tau);

/* ---------------------------------------------------------------------------
 * 40 Hz -> 100 Hz reference interpolation for B items (one item = one 3-vector quantity of one robot).  Replaces
 * PRMPCClass::XGetSolution_position_mod3 (RT/FastMPC/PRMPCClass.cpp:1170-1261, with _AAA_inv_mod of
 * solve_AAA_inv_mod1 :1344-1361) as rt_mpc_qp calls it per quantity (RT/gait_fast.cpp:131-138): the cubic through
 * four consecutive 40 Hz samples, evaluated at walktime * dt_sample + jx * dt_sample, jx = 0..nh-1.
 *   walktime_d [B] ints; samples_d [12][B]: in1 xyz | in2 xyz | ref xyz | ref2 xyz (SoA [f*B + b])
 *   out_d [9 + 3 (nh - 1)][B]: position, velocity, acceleration at jx = 0, then the positions at jx = 1..nh-1
 *   (the reference's Vec21 at its nh = 4); all zero once walktime > _t_end_footstep.
 * Parity (tests/test_zz_ref_interp.py, B200): 1e-9 relative to the pinned oracle (oracle/ref_interp.c; the reference
 * evaluates the monomials with libm pow, the kernel with a correctly rounded integer power), 1e-12 absolute over the
 * reference's own walktime range (count_inteplotation = 1..2, RT/gait_fast.cpp:113-131).
 * ------------------------------------------------------------------------ */
int go1mpc_ref_interp_batch(go1mpc_t *h, int B, int nh, const int *walktime_d, double dt_sample,
                            const double *samples_d, double *out_d, void *stream);
/* Host part, needs no device: _AAA_inv_mod (row-major 4x4) and _t_end_footstep (:179) for a configuration
 * (NULL = defaults); either output may be NULL. */
int go1mpc_ref_interp_model(const Go1MpcConfig *cfg, double *inv16, int *t_end_footstep);

/* ---------------------------------------------------------------------------
 * One control tick for B robots with HOST inputs and COMPACT results -- the call a controller farm makes per tick:
 * planner tick (= go1mpc_step_timing_step_batch) and body-inclination MPC tick on the device-resident records
 * (= go1mpc_body_mpc_step_batch_resident_host_async) on ONE caller stream, then a 12-double result row per robot.
 * What the reference classes keep as members stays in HBM (planner state, _tx, _V_ini / stale results); what their
 * tick methods take as arguments moves up per call (tick, the 20 -- or 10, see step_in_rows -- planner inputs, the 9+9nh
 * body-tick doubles); what
 * comes down is GO1MPC_COMPACT_DOUBLES per robot instead of Vec38 + Vec14 + diagnostics:
 *   [0,3) CoM x y z (Vec38 0..2)   [3,5) body roll, pitch   [5,7) body torques (Vec14 0..3)
 *   [7,9) next footstep x, y (Vec38 29, 31)   [9] step period (Vec38 35)
 *   [10] status of the planner's last SQP solve (-1: none ran)   [11] body QP status
 * compact_d is a caller-owned DEVICE buffer [B][12] (16-byte aligned; e.g. the send buffer of the once-per-batch gather
 * to rank 0); `compact` (host, may be NULL) receives a copy.  out38 / step_diag / body_diag (host, may be NULL) receive
 * the full results.  step_state_src_d (may be NULL): run the planner tick out of place from this pristine state.
 * Everything is enqueued on `stream`; staging is per stream and owned by the handle.
 * ------------------------------------------------------------------------ */
#define GO1MPC_COMPACT_DOUBLES 12
typedef struct {
  int n_sqp, nh;
  const int *tick;                /* host [B] */
  const double *step_in;          /* host [20][B] */
  const double *body_tick_in;     /* host [B][go1mpc_body_tick_in_stride(nh)] */
  const double *step_state_src_d; /* device [202][B] or NULL */
  double *step_state_d;           /* device [202][B], state after the tick */
  const double *tx_d;             /* device [B][28] */
  double *body_out_d;             /* device [B][go1mpc_body_out_stride(nh)], in/out */
  double *compact_d;              /* device [B][12] */
  double *compact;                /* host [B][12] or NULL */
  double *out38;                  /* host [38][B] or NULL */
  int *step_diag;                 /* host [60][B] or NULL */
  int *body_diag;                 /* host [B][go1mpc_body_diag_stride(nh)] or NULL */
  int step_in_rows;               /* leading rows of step_in that are uploaded: 0 or 20 = all; 10 = the sensor rows only
                                   * (estimated CoM state, foot locations; step_in is then host [10][B]).  Rows 10..19 -- the
                                   * external CoM-height samples (read only with cfg.step.ext_height) and the terrain heights
                                   * Zsc -- then read as zero: flat ground, the reference's own configuration */
} Go1ControlTick;
int go1mpc_control_tick_host_async(go1mpc_t *h, int B, const Go1ControlTick *t, void *stream);
/* The pack kernel alone (device pointers; step_diag_d / body_diag_d may be NULL). */
int go1mpc_pack_compact_batch(go1mpc_t *h, int B, int nh, const double *out38_d, const int *step_diag_d,
                              const double *body_out_d, const int *body_diag_d, double *compact_d, void *stream);

/* ---------------------------------------------------------------------------
 * Once-per-batch gather of result rows to rank 0 over NVLink / NVSwitch peer memory, without a collective (SURVEY 8e).
 * Rank 0 owns `slots` blocks [world][rows_per_rank][row_doubles]; it exports an IPC blob the host program hands to the
 * other ranks (one process per GPU); a peer maps the memory and lets its kernels write its rows straight into rank 0's
 * block: go1mpc_gather_dest() is a valid compact_d for go1mpc_control_tick_host_async.  Per use of a slot, all on a stream:
 *   peer:   acquire -> [tick writing to dest] -> publish
 *   rank 0: [tick writing to dest] -> publish -> wait_all -> [read go1mpc_gather_block, e.g. D2H] -> release
 * acquire / wait_all are single-thread device-side waits on flags in rank 0's memory (about 10 s time-out -> go1mpc_gather_status);
 * no rank ever waits for another on the host.  Every rank must use a slot the same number of times, in the same order.
 * ------------------------------------------------------------------------ */
typedef struct go1mpc_gather go1mpc_gather_t;
#define GO1MPC_GATHER_BLOB_BYTES 128
int go1mpc_gather_create(int device, int rank, int world, int slots, int rows_per_rank, int row_doubles, go1mpc_gather_t **out);
void go1mpc_gather_destroy(go1mpc_gather_t *g);
int go1mpc_gather_export(go1mpc_gather_t *g, void *blob, int blob_bytes);          /* rank 0 */
int go1mpc_gather_import(go1mpc_gather_t *g, const void *blob, int blob_bytes);    /* peers */
double *go1mpc_gather_dest(go1mpc_gather_t *g, int slot);
const double *go1mpc_gather_block(go1mpc_gather_t *g, int slot);                   /* rank 0 */
int go1mpc_gather_acquire(go1mpc_gather_t *g, int slot, void *stream);
int go1mpc_gather_publish(go1mpc_gather_t *g, int slot, void *stream);
int go1mpc_gather_wait_all(go1mpc_gather_t *g, int slot, void *stream);            /* rank 0 */
int go1mpc_gather_release(go1mpc_gather_t *g, int slot, void *stream);             /* rank 0 */
int go1mpc_gather_status(go1mpc_gather_t *g, int *status);

/* ---------------------------------------------------------------------------
 * Stream ordering and CUDA-graph capture.  Every *_batch entry only enqueues work on the stream it is given and
 * allocates nothing once that stream has been used with the same batch size, so a sequence of ticks dealt over several
 * streams can be captured once and replayed with one launch (launch-bound loops at small batches):
 *   go1mpc_graph_capture_begin(h, s0); go1mpc_stream_wait(h, s1, s0); ...ticks on s0, s1...;
 *   go1mpc_stream_wait(h, s0, s1); go1mpc_graph_capture_end(h, s0, &g); go1mpc_graph_launch(h, g, s0);
 * go1mpc_stream_wait makes `waiter` wait for the work enqueued so far on `signaller` (NULL = the handle's stream).
 * A handle keeps a workspace for at most 256 distinct streams; a call that would bring in a 257th returns
 * GO1MPC_E_UNSUPPORTED and enqueues nothing.
 * ------------------------------------------------------------------------ */
int go1mpc_stream_wait(go1mpc_t *h, void *waiter, void *signaller);
int go1mpc_graph_capture_begin(go1mpc_t *h, void *stream);
int go1mpc_graph_capture_end(go1mpc_t *h, void *stream, void **graph_exec_out);
int go1mpc_graph_launch(go1mpc_t *h, void *graph_exec, void *stream);
int go1mpc_graph_destroy(go1mpc_t *h, void *graph_exec);

/* ---------------------------------------------------------------------------
 * Signal filters of go1_servo's 1 kHz loop for B robots x C channels (SURVEY 8f-4).  Replaces butterworthLPF::filter
 * (GO1/Filter/butterworthLPF.cpp:104-121; init :82-100 = go1mpc_lpf_coefficients) -- 28 objects on slots of the /MPC/Gait
 * message, servo.cpp:579-610,898-931 -- and ButterworthFilter::ForceFilter (GO1/Filter/butterworth_filter.cpp:37-69).
 * coef      host, [C][6]: b0 b1 b2 a1 a2 a per channel (C <= 32 per call)
 * in_d      [rows][B] SoA; channel c filters row in_rows_d[c] (device ints) or row c when in_rows_d is NULL -- so the channels
 *           can be picked straight out of a [100][B] message buffer
 * state_d   [5][C][B] SoA, in/out: call counter, y_p, y_pp, x_p, x_pp of every filter object; zero-initialise
 *           (force filter: [6][C][B]: count, raw[2], filtered[3])
 * out_d     [C][B]
 * Bit-identical to the reference classes (tests/test_filters.py).
 * ------------------------------------------------------------------------ */
int go1mpc_lpf_coefficients(double fsampling, double fcutoff, double *coef6);
int go1mpc_lpf_batch(go1mpc_t *h, int B, int C, const double *coef, const double *in_d, const int *in_rows_d, double *state_d,
                     double *out_d, void *stream);
int go1mpc_force_filter_batch(go1mpc_t *h, int B, int C, const double *in_d, double *state_d, double *out_d, void *stream);

/* ---------------------------------------------------------------------------
 * The 40 Hz planner node of mosek_nlp_kmp for B robots: one call of NLPRTControlClass::WalkingReactStepping per robot,
 * /MPC/Gait message out.  Replaces NLP/NLPRTControl/NLPRTControlClass.cpp:191-396 (squat / walk / over / idle branches and the
 * 100-slot message layout :288-392), StartWalking / StopWalking :400-432, rt_nlp_gait :436-596 with everything it calls:
 *   NLPClass::X_CoM_position_squat (NLP/NLP/NLPClass_sqp.cpp:2958-3015), step_timing_opti_loop + CoM_height_solve,
 *   Foot_trajectory_solve_mod2 with its stop-walking branch, Zmp_distributor / zmp_interpolation / Force_torque_calculate
 *   (:3650-3897).
 * state_d     [go1mpc_nlp_node_state_doubles()][B] SoA, in/out: rows [0,202) the planner state, [202,234) the swing-foot
 *             window, then the ZMP ring and the node's members (go1mpc_nlp_node_default_state gives one robot's column)
 * walkdtime_d [B] ints: the caller's tick counter (the reference's walkdtime, 1, 2, 3 ...; the walk's ticks must be consecutive)
 * start_d     [B] ints or NULL (= 1): start_mpc;   cmd_d [B] ints or NULL: 1 = StopWalking(), 2 = StartWalking() before the tick
 * rfoot_fb_d / lfoot_fb_d  [3][B] or NULL (= 0): measured foot locations.  The reference ignores its estimated-state argument
 *             (rt_nlp_gait passes the all-zero member _estimated_state, :446), so there is none here.
 * msg_d       [100][B] SoA: the message (slot 98 = 0)
 * Six launches on `stream`.  Parity: tests/test_gpu_nlp_node.py (cfg1 and stop / restart scripts of the unmodified class).
 * ------------------------------------------------------------------------ */
/* rows of the node state a host may read or set between ticks (exact integers / flags stored as doubles) */
#define GO1MPC_NLP_ROW_STOP 365          /* _stop_walking */
#define GO1MPC_NLP_ROW_START_AGAIN 366   /* _start_walking_again */
#define GO1MPC_NLP_ROW_T_INT 367         /* _t_int: planner tick of the last walking call */
#define GO1MPC_NLP_ROW_MPC_STOP 368      /* mpc_stop */
#define GO1MPC_NLP_ROW_RIGHT_SUPPORT 369 /* right_support */
int go1mpc_nlp_node_state_doubles(void);
int go1mpc_nlp_node_default_state(go1mpc_t *h, double *state);
int go1mpc_nlp_walkdtime_max(const go1mpc_t *h);         /* _walkdtime_max: ticks of the walk (672) */
int go1mpc_nlp_t_end_footstep(const go1mpc_t *h);        /* _t_end_footstep */
int go1mpc_nlp_node_tick_batch(go1mpc_t *h, int B, double *state_d, const int *walkdtime_d, const int *start_d, const int *cmd_d,
                               const double *rfoot_fb_d, const double *lfoot_fb_d, double *msg_d, void *stream);
/* host buffers of the same SoA shapes (synchronous: copies up, tick, copies down) */
int go1mpc_nlp_node_tick_batch_host(go1mpc_t *h, int B, double *state, const int *walkdtime, const int *start, const int *cmd,
                                    const double *rfoot_fb, const double *lfoot_fb, double *msg);

/* ---------------------------------------------------------------------------
 * The 100 Hz node of rt_mpc_qp for B robots: /MPC/Gait message in, /rtMPC/traj message out.  Replaces one pass of the
 * main loop of RT/gait_fast.cpp:505-746 with everything it calls:
 *   xget_position_interpolation (:113-372) + PRMPCClass::XGetSolution_position_mod3 (RT/FastMPC/PRMPCClass.cpp:1170-1261),
 *   PRMPCClass::Foot_trajectory_solve_mod2 (:1756-2195), XGetSolution_Foot_rotation (:2255-2380), the 2 x nh reference
 *   windows (gait_fast.cpp:568-616, with their row-0-twice quirk), PRMPCClass::body_theta_mpc, the outgoing 100 slots
 *   (:633-729; slot 86 -- wall time -- is 0).
 * state_d  [go1mpc_rt_node_state_doubles(nh)][B] SoA, in/out: the node's and the class's members
 *          (go1mpc_rt_node_default_state gives one robot's initial column)
 * msg_d    [100][B] SoA: the latest message of the 40 Hz planner per robot (slots as NLPRTControlClass.cpp:288-392)
 * ctrl_d   [B] ints (control_gait(0) > 0) or NULL = on;  bodyangle_state_d [4][B] or NULL = 0
 * body_in_d  [B][go1mpc_body_in_stride(nh)] workspace; body_out_d [B][go1mpc_body_out_stride(nh)] the body MPC's records
 *          (in/out: its state lives there; zero-initialise);  body_diag_d as go1mpc_body_mpc_step_batch or NULL
 * out100_d [100][B] SoA;  active_d [B] ints or NULL: 1 where the fast tick ran (message slot 99 > 0)
 * Three launches on `stream`.  Parity: tests/test_gpu_rt_node.py (cfg1 lock-step replay of the unmodified classes).
 * ------------------------------------------------------------------------ */
int go1mpc_rt_node_state_doubles(int nh);
int go1mpc_rt_node_default_state(go1mpc_t *h, int nh, double *state);
int go1mpc_rt_node_tick_batch(go1mpc_t *h, int nh, int B, double *state_d, const double *msg_d, const int *ctrl_d,
                              const double *bodyangle_state_d, double *body_in_d, double *body_out_d, int *body_diag_d,
                              double *out100_d, int *active_d, void *stream);
/* The same tick with the node's other two topics in their wire format (gait_fast.cpp:92-110, 519-527): ctl_msg_d [25][B] is
 * /control2rtmpc/state -- slot 0 the control flag control_gait(0), slots 10, 11, 13, 14 the measured body angles / rates the
 * MPC is fed (bodyangle_state) --, rt2nrt_msg_d [25][B] (or NULL) receives /rt2nrt/state: slot 0 = t_int, slots 1..24 = the
 * control message's. */
int go1mpc_rt_node_tick_msgs_batch(go1mpc_t *h, int nh, int B, double *state_d, const double *gait_msg_d, const double *ctl_msg_d,
                                   double *body_in_d, double *body_out_d, int *body_diag_d, double *traj_msg_d,
                                   double *rt2nrt_msg_d, void *stream);
/* host buffers (synchronous); body_out [B][go1mpc_body_out_stride(nh)] is the body MPC's state, in/out */
int go1mpc_rt_node_tick_batch_host(go1mpc_t *h, int nh, int B, double *state, const double *msg, const int *ctrl,
                                   const double *bodyangle_state, double *body_out, double *out100);

/* ---------------------------------------------------------------------------
 * Gait stack tick: both nodes above behind ONE host call per 100 Hz tick for B robots that share one clock -- the call a
 * controller farm makes every 10 ms.  The sensor slots the nodes read go up, the result slots the servo consumes come down;
 * everything the reference keeps as node members (and both nodes' messages) stays in HBM, in one SoA state [row][B]:
 *   [GO1MPC_STACK_ROW_NLP, +go1mpc_nlp_node_state_doubles())   the planner node's state
 *   [GO1MPC_STACK_ROW_GAIT, +100)      /MPC/Gait                  [GO1MPC_STACK_ROW_RT2NRT, +25)  /rt2nrt/state
 *   GO1MPC_STACK_ROW_WALKDTIME         the planner's tick counter walkdtime (exact integer)
 *   [GO1MPC_STACK_ROW_TRAJ, +100)      /rtMPC/traj                [GO1MPC_STACK_ROW_RT, +go1mpc_rt_node_state_doubles(nh))  the 100 Hz node
 * go1mpc_gait_stack_default_state gives one robot's initial column; a robot is reset by rewriting its column, a batch is
 * checkpointed by a memcpy.  One call enqueues on `stream`:
 *   1. H2D of sensor (and, when planner = 1, of cmd / start if given); an input given as a device buffer (sensor_d, cmd_d,
 *      start_d) is read in place instead, with no copy
 *   2. planner = 1: walkdtime += 1, then go1mpc_nlp_node_tick_batch on the state with rfoot_fb / lfoot_fb = rows 22..24 / 19..21
 *      of the resident /rt2nrt/state (the foot feedback the previous fast tick forwarded, as the reference's ROS graph wires it)
 *   3. the sensor rows into their slots of a /control2rtmpc/state buffer (its other 14 slots 0), then
 *      go1mpc_rt_node_tick_msgs_batch writing /rtMPC/traj and /rt2nrt/state into the state
 *   4. the n_slots selected slots of both messages -> rows_d [B][n_slots]; D2H into rows when given
 * Results are bit-identical to calling the two node entries in that order.  The reference's clock (planner every 25 ms,
 * fast node every 10 ms): the fast tick at 10k ms sets planner = 1 when a multiple of 25 lies in (10(k-1), 10k], k = 0, 3, 5,
 * 8, 10, ...  The body-MPC input records and all staging are per-stream workspace owned by the handle, allocated on the
 * first call with a given (stream, B): later calls with that pair allocate nothing, so a warmed-up schedule can be captured
 * with go1mpc_graph_capture_*.  Host buffers should be pinned and stay untouched until the stream has passed the call.
 * Device inputs: sensor_d [11][B] (in place of sensor), cmd_d / start_d [B] (in place of cmd / start) give bit-identical
 * results to host inputs holding the same values.  They are read by the call's own kernels in stream order: a kernel enqueued
 * earlier on `stream` may write them and one enqueued after the call may overwrite them (a writer on another stream needs the
 * caller's events).  Device values are not checked: as for the host inputs, a cmd other than 1 or 2 is no command.
 * Errors (nothing is enqueued): GO1MPC_E_INVALID for a NULL required pointer, both or neither of sensor / sensor_d, both of
 * cmd / cmd_d or of start / start_d, n_slots outside 1..64, a slot outside 0..199, body_out_d not 16-byte, rows_d or sensor_d
 * not 8-byte, cmd_d or start_d not 4-byte aligned, a device input whose address range overlaps state_d, body_out_d, rows_d
 * (or the clocked tick's clock_d) -- the call's kernels take them as non-aliasing; GO1MPC_E_UNSUPPORTED for nh outside 3..40
 * or cfg.step.ext_height set.
 * ------------------------------------------------------------------------ */
#define GO1MPC_STACK_SENSOR_ROWS 11   /* /control2rtmpc/state slots 0 | 10 11 13 14 | 19 20 21 | 22 23 24 */
#define GO1MPC_STACK_SLOTS_MAX 64
#define GO1MPC_STACK_ROW_NLP 0
#define GO1MPC_STACK_ROW_GAIT 480
#define GO1MPC_STACK_ROW_RT2NRT 580
#define GO1MPC_STACK_ROW_WALKDTIME 605
#define GO1MPC_STACK_ROW_TRAJ 606
#define GO1MPC_STACK_ROW_RT 706
typedef struct {
  int nh;                    /* body-MPC horizon, 3..40 */
  int planner;               /* 1: the 40 Hz planner node ticks first in this call */
  const double *sensor;      /* host [11][B] SoA: control flag, body angles / rates, L foot xyz, R foot xyz */
  const int *cmd, *start;    /* host [B] or NULL; read only when planner = 1 (as go1mpc_nlp_node_tick_batch) */
  double *state_d;           /* device [go1mpc_gait_stack_state_doubles(nh)][B] SoA, in/out */
  double *body_out_d;        /* device [B][go1mpc_body_out_stride(nh)], in/out, zero-initialised, 16-byte aligned */
  int n_slots;
  int slots[GO1MPC_STACK_SLOTS_MAX];   /* 0..99 = /MPC/Gait slot, 100..199 = /rtMPC/traj slot - 100 */
  double *rows_d;            /* device [B][n_slots], caller-owned (e.g. go1mpc_gather_dest with row_doubles = n_slots) */
  double *rows;              /* host [B][n_slots] or NULL: copy of rows_d */
  const double *sensor_d;    /* device [11][B] SoA, same rows as `sensor`; exactly one of sensor / sensor_d */
  const int *cmd_d, *start_d;  /* device [B] or NULL; at most one of cmd / cmd_d and one of start / start_d */
} Go1GaitStackTick;
int go1mpc_gait_stack_state_doubles(int nh);
int go1mpc_gait_stack_default_state(go1mpc_t *h, int nh, double *column);
int go1mpc_gait_stack_tick_host_async(go1mpc_t *h, int B, const Go1GaitStackTick *t, void *stream);

/* ---------------------------------------------------------------------------
 * Gait stack with per-robot clocks and on-device resets: one batch holds robots at arbitrary points of their episodes (Monte-Carlo /
 * RL farms), and each robot's run is bit-identical to a fresh run of that robot started at its reset.
 *
 * go1mpc_gait_stack_tick_clocked_async: go1mpc_gait_stack_tick_host_async with the planner flag taken per robot from
 *   clock_d  device [B] ints, in/out, caller-owned: 10 ms periods since the robot's reset (zero-initialise a fresh batch).
 *   Robot b with clock c plans in this call when c == 0 or (10c)/25 > (10(c-1))/25 (c = 0, 3, 5, 8, 10, ...: the reference's
 *   schedule, run on the robot's own time); its clock is c + 1 after the call.  walkdtime += 1 only for the robots that plan.  A robot
 *   that does not plan leaves the planner node's rows, /MPC/Gait and walkdtime untouched; the 100 Hz node, the pack and the copy to
 *   `rows` run for every robot.  cmd / start are uploaded whenever given (cmd_d / start_d are read in place) and read only for
 *   the robots that plan; sensor_d / cmd_d / start_d as go1mpc_gait_stack_tick_host_async.  The planner node's
 *   kernels are enqueued on every call (robots that do not plan exit at once), so every call enqueues the same work and one captured
 *   period graph replays for all periods.  Errors: those of go1mpc_gait_stack_tick_host_async, and GO1MPC_E_INVALID for a NULL
 *   clock_d; nothing is enqueued on an error.  B = 0 is a no-op.
 *
 * go1mpc_gait_stack_reset_async: for every robot b with reset[b] != 0 (reset: host [B] ints, pinned so the call can sit in a graph,
 *   uploaded by the call; or reset_d: device [B] ints read in place in stream order, as the ticks' device inputs):
 *     the column b of state_d = go1mpc_gait_stack_default_state(nh);  body_out_d record b = 0;  clock_d[b] = 0;
 *     when servo_state_d is given: rows GO1MPC_SERVO_ROW_Q..+12 = servo_q0, the 45 filter rows = 0 (the homing rows are the
 *     caller's input and stay).
 *   Other robots are not touched.  Two kernel launches of a fixed shape; the flagged robots are listed on the device, so the
 *   flags never change what is enqueued, and the work grows with the number of robots flagged.  The default column is built once
 *   per (handle, nh), with a synchronous upload, and kept on the device: the first reset call with each nh must come before any
 *   graph capture.  Any non-zero flag resets the robot.  Errors (nothing is enqueued): GO1MPC_E_INVALID for both or neither of
 *   reset / reset_d, a NULL clock_d / state_d / body_out_d, body_out_d not 16-byte or reset_d not 4-byte aligned, reset_d
 *   overlapping state_d, body_out_d, clock_d or servo_state_d; GO1MPC_E_UNSUPPORTED for nh outside 3..40.
 *
 * Both entries allocate only on their first call with a given (stream, B) (and, for the reset, nh), so a warmed-up period
 *   reset -> clocked tick -> go1mpc_servo_stack_tick_async can be captured once with go1mpc_graph_capture_* and replayed every period.
 *   Fed from host buffers, the caller rewrites the pinned sensor and reset buffers between replays, after the previous replay has
 *   finished.  Fed from device buffers -- sensor_d, cmd_d / start_d, reset_d (or a restart by go1mpc_farm_copy_async), with the
 *   optional host copies (rows, and the servo entries' q / tau) left NULL -- a period enqueues no host<->device copy: a simulator
 *   kernel on the same stream writes the next period's inputs, and periods are enqueued or replayed back to back with no host
 *   synchronisation.
 * ------------------------------------------------------------------------ */
typedef struct {
  int nh;                    /* body-MPC horizon, 3..40 */
  const double *sensor;      /* host [11][B] SoA, as Go1GaitStackTick */
  const int *cmd, *start;    /* host [B] or NULL; read only for the robots that plan in this call */
  double *state_d;           /* device [go1mpc_gait_stack_state_doubles(nh)][B] SoA, in/out */
  double *body_out_d;        /* device [B][go1mpc_body_out_stride(nh)], in/out, zero-initialised, 16-byte aligned */
  int n_slots;
  int slots[GO1MPC_STACK_SLOTS_MAX];   /* as Go1GaitStackTick */
  double *rows_d;            /* device [B][n_slots] */
  double *rows;              /* host [B][n_slots] or NULL */
  int *clock_d;              /* device [B] ints, in/out: periods since each robot's reset */
  const double *sensor_d;    /* as Go1GaitStackTick */
  const int *cmd_d, *start_d;  /* as Go1GaitStackTick */
} Go1GaitStackClockedTick;
int go1mpc_gait_stack_tick_clocked_async(go1mpc_t *h, int B, const Go1GaitStackClockedTick *t, void *stream);
typedef struct {
  int nh;
  const int *reset;          /* host [B] ints (pinned) or NULL: non-zero = reset this robot */
  int *clock_d;              /* device [B], as Go1GaitStackClockedTick */
  double *state_d;           /* device [go1mpc_gait_stack_state_doubles(nh)][B] */
  double *body_out_d;        /* device [B][go1mpc_body_out_stride(nh)], 16-byte aligned */
  double *servo_state_d;     /* device [GO1MPC_SERVO_STATE_ROWS][B] or NULL */
  double servo_q0[12];       /* joint angles (FR, FL, RR, RL) a reset robot's servo starts from */
  const int *reset_d;        /* device [B] ints, same flags as `reset`; exactly one of reset / reset_d */
} Go1GaitStackReset;
int go1mpc_gait_stack_reset_async(go1mpc_t *h, int B, const Go1GaitStackReset *r, void *stream);

/* ---------------------------------------------------------------------------
 * Farm column copy: whole robots copied between two farm-shaped buffer sets, the source column picked per destination column by
 * a device index array -- to snapshot robots into a bank, restore them, fork one stored mid-walk state into many robots, or
 * restart robots chosen by a device kernel (a simulator's episode end) with no host round trip.
 *
 * A robot's whole state is its gait stack column state_d[:, b], its body-MPC record body_out_d[b], its clock clock_d[b], its
 * servo column servo_state_d[:, b] and its force column force_state_d[:, b]: a run that starts from copied values is
 * bit-identical to the run of the robot they were copied from.  For every destination column i with 0 <= index_d[i] < src.B,
 * every given block of column i becomes the same block of source column index_d[i].  The servo column is copied whole, homing
 * rows included (go1mpc_gait_stack_reset_async keeps them).  index_d[i] = -1 keeps column i; any other entry outside
 * -1..src.B-1 also keeps column i and, when bad_d is given, adds 1 to *bad_d.  Each destination has one source, so there are no
 * write conflicts; many destinations may share one source.  The same call serves
 *   snapshot  farm -> bank    (dst = a bank of any B, index_d[j] = the farm column to store in bank column j)
 *   restore   bank -> farm    (index_d[i] = the bank column robot i restarts from, -1 for robots that keep walking)
 *   fork      bank -> farm with a repeated index (one stored state into many robots), or farm A -> farm B
 * A fork inside one farm is two calls through a bank: snapshot robot 7 into bank column 0 (bank index {7}), then restore with
 * index_d[i] = 0 for the robots that fork and -1 elsewhere.  A bank column holding a freshly reset robot (snapshot right after
 * go1mpc_gait_stack_reset_async, force column zero) restarts robots as that reset plus the torque tick's reset flag do, except
 * that the homing rows come from the bank column.
 * clock_d, servo_state_d, force_state_d and health_d are each given on both sides or on neither; both sides share nh.
 * health_d (the farm's health counters, see go1mpc_gait_stack_tick_clocked_health_async) travels with the clock: a copied
 * column takes the source's counters, so a snapshot and restore continues counting bit-identically.  A restore given no health
 * block leaves the destination's old counters in place; they restart anyway when the restored clock is 0 (the next health-enabled
 * clocked tick zeroes them).
 * Two kernel launches of a fixed shape after a memset of a device counter: the first lists the copied destinations (one
 * atomic per warp) and copies their clocks, the second copies the listed columns, reading the count on the device.  The index
 * never changes what is enqueued, and the work grows with the number of columns copied.  A workspace of 8 B per destination
 * column is allocated on the first call with a given (stream, dst.B); later calls allocate nothing, so a warmed-up period
 * restore -> go1mpc_gait_stack_tick_clocked_async -> go1mpc_servo_torque_tick_async can be captured once with
 * go1mpc_graph_capture_* and replayed, the caller (or a device kernel) rewriting index_d between replays.  dst.B = 0 is a no-op.
 * Errors (nothing is enqueued): GO1MPC_E_INVALID for a NULL c, state_d, body_out_d or index_d, an optional block given on one
 * side only, body_out_d not 16-byte or health_d not 4-byte aligned on either side, a negative B, src.B < 1 while dst.B > 0, or any destination block
 * whose address range overlaps any source block; GO1MPC_E_UNSUPPORTED for nh outside 3..40.  index_d is device memory and is
 * not checked on the host: an out-of-range entry never causes an out-of-bounds access.
 * ------------------------------------------------------------------------ */
typedef struct {
  int B;                    /* columns (robots) of this buffer set */
  double *state_d;          /* [go1mpc_gait_stack_state_doubles(nh)][B] SoA */
  double *body_out_d;       /* [B][go1mpc_body_out_stride(nh)], 16-byte aligned */
  int *clock_d;             /* [B] or NULL */
  double *servo_state_d;    /* [GO1MPC_SERVO_STATE_ROWS][B] or NULL */
  double *force_state_d;    /* [GO1MPC_SERVO_FORCE_ROWS][B] or NULL */
  int *health_d;            /* [GO1MPC_HEALTH_ROWS][B] ints, 4-byte aligned, or NULL */
} Go1FarmColumns;
typedef struct {
  int nh;                   /* 3..40, shared by both sides */
  Go1FarmColumns dst, src;
  const int *index_d;       /* device [dst.B]: -1 = keep column i; 0..src.B-1 = column i <- source column index_d[i] */
  int *bad_d;               /* device int or NULL: += number of entries outside -1..src.B-1 (those columns are kept) */
} Go1FarmCopy;
int go1mpc_farm_copy_async(go1mpc_t *h, const Go1FarmCopy *c, void *stream);

/* ---------------------------------------------------------------------------
 * Servo stack tick: K consecutive ticks of go1_servo's 1 kHz loop for B robots in ONE call, fed in place from the messages the
 * gait stack keeps resident -- the call a controller farm makes after each gait stack call (K = 10 per 10 ms period), joint
 * targets out.  Per robot b and tick k = 1..K:
 *   filters   9 butterworthLPF objects, go1mpc_lpf_coefficients(1000, 3), on /MPC/Gait slots 0 1 2 6 7 8 9 10 11 (channels
 *             0..8 in that order), each stepped once per tick on the held message value -- as 9 objects called every 1 kHz tick
 *   IK        go1mpc_servo_kin_tick_batch's leg mapping and 4 x Inverse_kinematics_g (servo.cpp:935-1051) with
 *               body position = filtered (slot 0, slot 1 * y_offset, slot 2)
 *               roll, pitch   = /rtMPC/traj slots 72, 73 (the body MPC's Vec14 [0], [1]), yaw 0 -- the fused tick's wiring
 *               left / right virtual foot = filtered slots 6 7 8 / 9 10 11
 *               initial guess = the previous tick's joint angles
 *             gait_mode (101 pace, 102 trot, 103 gallop) and y_offset as in go1mpc_servo_kin_tick_batch
 * The result equals K x (go1mpc_lpf_batch on the state's /MPC/Gait block + go1mpc_servo_kin_tick_batch) bit for bit.
 * Servo state, caller-owned SoA [GO1MPC_SERVO_STATE_ROWS][B]:
 *   [GO1MPC_SERVO_ROW_Q, +12)       joint angles q (FR, FL, RR, RL), in/out
 *   [GO1MPC_SERVO_ROW_HOMING, +12)  homing foot positions (input, as go1mpc_servo_kin_tick_batch's homing_d)
 *   [GO1MPC_SERVO_ROW_LPF, +45)     the 9 filters' state in go1mpc_lpf_batch's [5][C][B] layout, C = 9; zero-initialise
 * A robot is reset by rewriting its column, a batch is checkpointed by a memcpy.
 * Not included: the servo's other filter objects (/MPC/Gait 39-41 and 73-75 at 10 Hz, ...) -- their outputs feed nothing here
 * and go1mpc_lpf_batch runs them on the resident message --, FK of the measured joints (servo.cpp:734-741), the GRF QP and
 * the torque map: go1mpc_servo_torque_tick_async below adds those three with its documented wiring.
 * One kernel launch, plus the D2H copy of q_d when q is given; nothing is allocated, so a warmed-up gait stack + servo period
 * can be captured with go1mpc_graph_capture_*.  B = 0 is a no-op.
 * Errors (nothing is enqueued): GO1MPC_E_INVALID for a NULL required pointer, K outside 1..GO1MPC_SERVO_TICKS_MAX, q_d not
 * 8-byte aligned; GO1MPC_E_UNSUPPORTED for gait_mode outside 101..103.
 * ------------------------------------------------------------------------ */
#define GO1MPC_SERVO_TICKS_MAX 10
#define GO1MPC_SERVO_STATE_ROWS 69
#define GO1MPC_SERVO_ROW_Q 0
#define GO1MPC_SERVO_ROW_HOMING 12
#define GO1MPC_SERVO_ROW_LPF 24
typedef struct {
  int K;                        /* 1..GO1MPC_SERVO_TICKS_MAX consecutive 1 kHz ticks */
  int gait_mode;
  double y_offset;
  const double *stack_state_d;  /* the gait stack's state [go1mpc_gait_stack_state_doubles(nh)][B], read only
                                   (/MPC/Gait at GO1MPC_STACK_ROW_GAIT, /rtMPC/traj at GO1MPC_STACK_ROW_TRAJ) */
  double *servo_state_d;        /* [GO1MPC_SERVO_STATE_ROWS][B] in/out */
  double *q_d;                  /* device [B][12*K]: per robot, tick-major joint targets (usable as a gather dest) */
  double *q;                    /* host [B][12*K] or NULL: D2H copy */
  double *jac_d, *foot_des_d;   /* last tick's [36][B] / [12][B], or NULL */
  int *iters_d;                 /* last tick's Newton updates [4][B], or NULL */
} Go1ServoStackTick;
int go1mpc_servo_stack_tick_async(go1mpc_t *h, int B, const Go1ServoStackTick *t, void *stream);

/* ---------------------------------------------------------------------------
 * Servo torque tick: go1mpc_servo_stack_tick_async's K ticks, each followed by the rest of go1_servo's 1 kHz tick
 * (servo.cpp: force_distribution / force_opt -> 4 x compute_joint_torques) -- joint targets AND feed-forward joint torques for
 * a Go1 in torque mode, with every member of Dynamiccclass resident on the device.  Per robot b and tick k = 1..K, after the
 * tick's filters and IK (identical to go1mpc_servo_stack_tick_async: q_d, the servo state, jac_d / foot_des_d / iters_d are
 * bit-identical to that call's):
 *   argument of the reference             source
 *   com_des, base_p                       the IK's body position of tick k (filtered slots 0, 1 * y_offset, 2)
 *   leg_des, leg_p, p_des                 the four IK foot targets of tick k (go1mpc_servo_stack_tick_async's foot_des_d)
 *   rfoot_des / lfoot_des                 the filtered virtual feet (filter channels 6-8 / 3-5)
 *   F_force_des                           /MPC/Gait 15-20 (F_L xyz, F_R xyz, force_distribution's order)
 *   FT_total_des                          (F_L + F_R, M_L + M_R) from /MPC/Gait 15-26
 *   right_support                         /MPC/Gait 99
 *   swing flag of leg l                   bit l of the QP's zero-force rule (mode 102: right_support 0 -> FL RR, 1 -> FR RL;
 *                                         mode 101: 0 -> FL RL, 1 -> FR RR; otherwise none)
 *   Jaco                                  the IK Jacobian at the tick's joint angles (the fused tick's wiring)
 *   p_est, pv_est                         FK of the measured joints with tick k's body pose (the planned pose: there is no
 *                                         estimator) = go1mpc_leg_fk_batch with body_r (roll, pitch, 0); pv_est_i =
 *                                         (J_i0 dq_0 + J_i1 dq_1) + J_i2 dq_2 with the measured-joint Jacobian J, no FMA
 *   pv_des                                /MPC/Gait 46-48 (right foot) / 49-51 (left foot), picked by the leg's virtual foot
 *   stance force in the torque map        the QP's grf_opt, or F_leg_guess when the QP returns NaN (the fused tick's wiring)
 * force_distribution runs for gait modes 101 / 102; mode 103 holds F_leg_ref (Dynamiccclass leaves it as it is).  The QP
 * (go1mpc_grf_force_opt_batch's constants) starts from the previous tick's grf_opt, so the K ticks chain.  Each tick equals
 * go1mpc_grf_force_distribution_batch -> go1mpc_grf_force_opt_batch -> go1mpc_grf_joint_torques_batch on records built as
 * above, bit for bit.
 * Buffers (device unless noted):
 *   force_state_d  [GO1MPC_SERVO_FORCE_ROWS][B] in/out, caller-owned, zero-initialise: rows [0,12) the previous tick's
 *                  grf_opt, rows [12,24) F_leg_ref (FR, FL, RR, RL xyz)
 *   meas_d         [24][B] measured joint angles (FR, FL, RR, RL) then joint velocities; sampled once per call and held over
 *                  its K ticks, as the messages are (K = 1 gives feedback every tick).  A host caller uploads it itself.
 *   reset          host [B] ints (pinned) or NULL: robots with a non-zero flag start from a zero force state -- the buffer
 *                  go1mpc_gait_stack_reset_async takes, so reset -> clocked tick -> torque tick replays with one set of flags
 *   reset_d        device [B] ints or NULL: the same flags read in place in stream order (at most one of reset / reset_d);
 *                  with reset_d, q = tau = NULL and the gait stack fed from device buffers, a period enqueues no
 *                  host<->device copy and runs back to back with a simulator kernel on the same stream
 *   tau_d          [B][12*K] joint torques, tick-major per robot like q_d;  tau: host [B][12*K] or NULL (D2H copy)
 *   grf_d, grf_diag_d  [B][16] / [B][32] or NULL: the last tick's out / diag records in go1mpc_grf_force_opt_batch's layout
 * Two kernel launches (the servo stack, then one warp per robot for the K force stages), plus the reset upload and the D2H
 * copies when given.  A workspace of 720 B per robot is allocated on the first call with a given (stream, B); later calls
 * allocate nothing and can be captured with go1mpc_graph_capture_*.  B = 0 is a no-op.
 * Errors (nothing is enqueued): GO1MPC_E_INVALID for a NULL required pointer (stack_state_d, servo_state_d, q_d,
 * force_state_d, meas_d, tau_d), K outside 1..GO1MPC_SERVO_TICKS_MAX, q_d or tau_d not 8-byte aligned, both reset and reset_d,
 * reset_d not 4-byte aligned or overlapping force_state_d, servo_state_d, q_d or tau_d; GO1MPC_E_UNSUPPORTED for gait_mode
 * outside 101..103.
 * ------------------------------------------------------------------------ */
#define GO1MPC_SERVO_FORCE_ROWS 24
typedef struct {
  int K;                        /* as Go1ServoStackTick */
  int gait_mode;
  double y_offset;
  const double *stack_state_d;
  double *servo_state_d;
  double *q_d;
  double *q;
  double *jac_d, *foot_des_d;
  int *iters_d;
  double y_coefficient;         /* force_distribution's y_coefficient */
  double *force_state_d;        /* [GO1MPC_SERVO_FORCE_ROWS][B] in/out */
  const double *meas_d;         /* [24][B] */
  const int *reset;             /* host [B] (pinned) or NULL */
  double *tau_d;                /* [B][12*K] */
  double *tau;                  /* host [B][12*K] or NULL */
  double *grf_d;                /* [B][16] or NULL */
  int *grf_diag_d;              /* [B][32] or NULL */
  const int *reset_d;           /* device [B] or NULL, same flags as `reset`; at most one of reset / reset_d */
} Go1ServoTorqueTick;
int go1mpc_servo_torque_tick_async(go1mpc_t *h, int B, const Go1ServoTorqueTick *t, void *stream);

/* ---------------------------------------------------------------------------
 * Farm health counters: per robot, how its solvers ended since the robot's reset, counted on the device by the farm's own kernels,
 * so that a Monte-Carlo or RL study can tell which robots drove a QP infeasible and how often, and restart robots whose controller
 * failed (go1mpc_farm_copy_async with an index computed on the device from the EVENTS row) with no host round trip.
 *
 * health_d: caller-owned device ints [GO1MPC_HEALTH_ROWS][B], SoA like every other farm block, zero-initialised; row r of robot b at
 * health_d[r * B + b].  Each row counts:
 *   PLAN_OK / _INFEASIBLE / _FAILED   planner SQP QPs (3 per planner tick) with status GO1MPC_QP_OK, GO1MPC_QP_INFEASIBLE, any other
 *                                     status >= 1 (NOT_PD, ITER_CAP, NAN, EQ_DEPENDENT); iterations that ran no solve count nowhere
 *   BODY_OK / _INFEASIBLE / _FAILED   the same split for body-MPC solves, one per clocked tick; a gated tick (status -1) counts nowhere
 *   GRF_OK / GRF_FAILED               servo ticks whose force QP returned GO1MPC_QP_OK / any other status (x = 0 is always feasible
 *                                     for that QP, so there is no infeasible row)
 *   GRF_FALLBACK                      servo ticks whose QP solution held a NaN, so the torque map used F_leg_guess (diag word 6 = 0)
 *   IK_CAP                            leg-ticks whose Inverse_kinematics_g applied all 15 updates (its stop test never passed)
 *   NONFINITE                         clocked ticks whose rows_d row of the robot holds a non-finite value, plus servo ticks whose
 *                                     12 q or 12 tau of the robot hold one
 *   EVENTS                            bit r (r = 0..10) set when row r grew during the current period: the clocked tick overwrites
 *                                     this row, the torque tick ORs into it
 * Counters restart with the robot's episode: a robot whose clock is 0 at the start of a health-enabled clocked tick starts that
 * call from zero (a fresh batch, a robot flagged by go1mpc_gait_stack_reset_async, a robot restored from a freshly reset bank
 * column).  clock_d counts the periods since that reset.  int32 is enough: IK_CAP, the fastest row, grows by at most 40 per period,
 * which takes more than 600 days of 100 Hz periods to overflow.
 *
 * go1mpc_gait_stack_tick_clocked_health_async: go1mpc_gait_stack_tick_clocked_async plus the counting.  The planner writes its step
 *   diag and the body MPC its diag records into a per-stream workspace (allocated with the other workspaces on the first call with
 *   a given (stream, B, nh)), and one more kernel after the pack updates health_d: planner rows for the robots that planned in this
 *   call, body rows for every robot, NONFINITE, the clock-0 restart and EVENTS.
 * go1mpc_servo_torque_tick_health_async: go1mpc_servo_torque_tick_async plus the counting of IK_CAP (in the servo stack kernel),
 *   the force-QP rows, GRF_FALLBACK and NONFINITE (in the force-stage kernel), tick by tick over the K ticks.  Same two launches.
 * With health, every output of both calls is bit-identical to the same call without it; the entries without health enqueue the
 * same work as before.  A warmed-up period restore -> clocked health tick -> torque health tick captures and replays as the plain one.
 * Errors (nothing is enqueued): those of the entry without health, and GO1MPC_E_INVALID for a NULL health_d, health_d not 4-byte
 * aligned, or a health_d range that overlaps a block the call reads or writes -- clocked tick: state_d, body_out_d, rows_d,
 * clock_d, sensor_d, cmd_d, start_d; torque tick: stack_state_d (its rows before GO1MPC_STACK_ROW_RT), servo_state_d,
 * force_state_d, meas_d, q_d, tau_d, reset_d, grf_d, grf_diag_d, jac_d, foot_des_d, iters_d.
 * Not covered: the position-mode farm entries go1mpc_gait_stack_tick_host_async and go1mpc_servo_stack_tick_async.
 * ------------------------------------------------------------------------ */
#define GO1MPC_HEALTH_ROWS 12
#define GO1MPC_HEALTH_PLAN_OK 0
#define GO1MPC_HEALTH_PLAN_INFEASIBLE 1
#define GO1MPC_HEALTH_PLAN_FAILED 2
#define GO1MPC_HEALTH_BODY_OK 3
#define GO1MPC_HEALTH_BODY_INFEASIBLE 4
#define GO1MPC_HEALTH_BODY_FAILED 5
#define GO1MPC_HEALTH_GRF_OK 6
#define GO1MPC_HEALTH_GRF_FAILED 7
#define GO1MPC_HEALTH_GRF_FALLBACK 8
#define GO1MPC_HEALTH_IK_CAP 9
#define GO1MPC_HEALTH_NONFINITE 10
#define GO1MPC_HEALTH_EVENTS 11
int go1mpc_gait_stack_tick_clocked_health_async(go1mpc_t *h, int B, const Go1GaitStackClockedTick *t, int *health_d, void *stream);
int go1mpc_servo_torque_tick_health_async(go1mpc_t *h, int B, const Go1ServoTorqueTick *t, int *health_d, void *stream);

/* Per-kernel timing of the three-launch body tick (measurement aid for bench.py's roofline): while enabled, each
 * go1mpc_body_mpc_step_batch call on that path records CUDA events around its setup / solve / merge launches;
 * go1mpc_body_phase_ms waits for the last such call and returns the three durations in milliseconds.  Do not enable
 * inside a graph capture. */
int go1mpc_body_phase_timing(go1mpc_t *h, int enable);
int go1mpc_body_phase_ms(go1mpc_t *h, float *ms3);

/* Measured FP64 FMA throughput of the device (GFLOP/s, 2 flop per FMA) from a
 * register-resident DFMA loop: the roofline denominator bench.py reports
 * against (SURVEY.md section 8d).  Runs ~`ms` milliseconds. */
int go1mpc_measure_dfma_peak(go1mpc_t *h, int ms, double *gflops);

#ifdef __cplusplus
}
#endif
#endif /* GO1MPC_H */
