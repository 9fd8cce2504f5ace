// kernels.h -- internal interface between the C-ABI host layer (api.cu) and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

namespace go1 {

struct BodyKParams {
  int nh, B;
  int in_stride, out_stride, diag_stride;   // doubles, doubles, ints
  int tab_doubles, warp_doubles;
  int cap_scale, gate, nstepx, nsum_mpc;
  const double* in;
  double* out;
  int* diag;
  const double* tab;
  int* sched;          // body_fast / body_split: {next instance, warps finished}, zero between launches
  // body_split appends the instances it hands to the combined kernel to flist (count in *flist_count);
  // body_fast with flist != null runs in list mode: it processes flist[0 .. *flist_count) -- or all B
  // instances when the count exceeded flist_cap -- and zeroes the count when its last warp leaves
  int* flist;
  int* flist_count;
  int flist_cap;
  // body_tri workspace (per stream): J per instance, state / result records per half, queue of active halves
  double *tri_jb, *tri_hs, *tri_res;
  int *tri_queue, *tri_qctl;      // qctl: {queued, fetched, guard trips, instances listed for the merge kernel}
  int* tri_meta;                  // compact list of the instances the merge kernel finishes (count: tri_qctl[3])
  double* tri_fr;                 // per instance: what the merge kernel needs of the input record
  double dt_mpc, j_ini, mass, g, gama, theta_lim, torque_lim;
  double lamda[4];
};
size_t body_smem_bytes(int nh, int wpc, int in_stride, int out_stride, int tab_doubles, int* warp_doubles);
cudaError_t body_mpc_launch(BodyKParams P, int wpc, int grid, size_t smem, cudaStream_t st);
cudaError_t body_mpc_occupancy(int wpc, size_t smem, int* blocks_per_sm);
// any horizon, roll / pitch halves interleaved in one warp (body_duo.cu); rare corners go to flist for body_mpc_launch
size_t body_duo_smem_bytes(int nh, int wpc, int in_stride, int out_stride, int* warp_doubles);
cudaError_t body_duo_launch(BodyKParams P, int sms, size_t smem_optin, cudaStream_t st);
// compile-time-horizon kernel (body_fast.cu); in/out strides and the table size must be the ABI's
bool body_fast_supported(int nh);
cudaError_t body_fast_launch(BodyKParams P, int sms, cudaStream_t st);
// roll / pitch halves side by side (body_split.cu); instances it cannot reproduce go to flist
// three launches, register-resident solver state (body_tri.cu)
bool body_tri_supported(int nh);
size_t body_tri_workspace_bytes(int nh, int B, size_t off[6]);   // offsets: J | half state | half result | queue | meta | hand-over
cudaError_t body_tri_launch(BodyKParams P, const double* tab_host, int sms, cudaStream_t st, cudaEvent_t* phase_ev = nullptr);
bool body_split_supported(int nh);
cudaError_t body_split_launch(BodyKParams P, int sms, cudaStream_t st);

struct DenseKParams {
  int n, p, m, B, cap;
  const double *G, *g0, *CE, *ce0, *CI, *ci0;
  double *x, *cost;
  int *active, *nactive, *iters, *status;
};
size_t dense_smem_bytes(int n, int m, int wpc);
cudaError_t dense_qp_launch(DenseKParams P, int wpc, int grid, size_t smem, cudaStream_t st);
cudaError_t dense_qp_occupancy(int wpc, size_t smem, int* blocks_per_sm);

// ---- step-location / step-timing SQP (step_timing.cu) ----
constexpr int STEP_STATE_DOUBLES = 202, STEP_IN_DOUBLES = 20, STEP_OUT_DOUBLES = 38;
constexpr int STEP_MAX_SQP = 5, STEP_DIAG_HEAD = 5, STEP_DIAG_PER = 11;
constexpr int STEP_DIAG_INTS = STEP_DIAG_HEAD + STEP_MAX_SQP * STEP_DIAG_PER;
struct StepCfgDev {
  double dt, Wn, ggg, t_min, t_max, footx_max, footx_min, footx_vmax, footx_vmin, footy_vmax, footy_vmin;
  double comax_max, comax_min, comay_max, comay_min, aax, aay, aaxv, aayv, bbx, bby, rr1, rr2;
  double half_hip_width, foot_width, lamda[4], hcom;
  double sh_dt, ch_dt, sh_w[3], ch_w[3];   // sinh / cosh(Wn dt) and (Wn dt jxx), jxx = 1..3: host libm, instance-independent
  int ext_height;
};
struct StepKParams {
  int B, n_sqp, cap;
  const int* tick;
  const double* state;  // [STEP_STATE_DOUBLES][B], state before the tick
  double* state_out;    // state after the tick; may alias `state` (in-place)
  const double* in;     // [STEP_IN_DOUBLES][B]
  double* out;          // [STEP_OUT_DOUBLES][B]
  int* diag;            // [STEP_DIAG_INTS][B] or null
  double* hz_co;        // [8][B] or null: the CoM-height polynomial of the tick (7 coefficients, highest power first) and the
                        //   sample index its time starts at -- for callers that evaluate samples beyond i + 2 (nlp_chain.cu)
  double* lipm;         // [6][B] or null: isx, visx, isy, visy, px, py of the LIPM roll-out (:896-901)
  const double* trtab;  // [STEP_TRTAB_ROWS][4]: cosh / sinh of Wn (t_min - k dt) (floored at 0.001 s) and of Wn (t_max - k dt), k = row
  StepCfgDev cfg;
};
constexpr int STEP_TRTAB_ROWS = 64;
// per-warp shared memory of the warp-cooperative mode: QP workspace (n = 4, m = 24) | 7x14 matrix + 7
constexpr int STEP_WARP_DOUBLES = 256;
cudaError_t step_timing_launch(StepKParams P, cudaStream_t st);   // step_timing.cu: warp per planner (small batches)
// step_sqp.cu: thread per planner, three launches (SQP, CoM height, back-end; the back-end expects state_out to hold a copy of state)
cudaError_t step_sqp_launch(StepKParams P, cudaStream_t st);
cudaError_t step_height_launch(StepKParams P, cudaStream_t st);
cudaError_t step_post_launch(StepKParams P, cudaStream_t st);
constexpr int FOOT_STATE_DOUBLES = 32, FOOT_OUT_DOUBLES = 18;
struct FootKParams {
  int B;
  const int* tick;
  const double* state;   // planner state AFTER the step-timing tick, [STEP_STATE_DOUBLES][B]
  const double* out38;   // its output ([38][B]): field 27 = _bjxx
  double* foot;          // [FOOT_STATE_DOUBLES][B], in/out
  double* out18;         // [18][B]
  int* right_support;    // [B] or null
  double dt, stepwidth0, lift_height;
  // stop-walking branch (:2043-2048), optional: lift0 [B] in/out = first step index whose lift height is zeroed (27 = none),
  // stop [B] = the caller's _stopwalking flag (non-zero = set); t_end = _t_end_footstep
  double* lift0;
  const double* stop;
  int t_end;
};
cudaError_t foot_traj_launch(FootKParams P, cudaStream_t st);

// ---- leg kinematics (leg_kin.cu); all arrays SoA [field][B] ----
struct LegKParams {
  int B;
  const double* q_in;     // FK: joint angles; IK: initial guess
  const int* leg;         // 0 FR, 1 FL, 2 RR, 3 RL
  const double* body_p;   // null = hip-frame variant
  const double* body_r;
  const double* pdes;     // IK target
  double* pos_out;        // FK
  double* q_out;          // IK
  double* jac_out;        // [9][B] row-major 3x3, may be null
  int* iters;             // IK updates applied, may be null
};
cudaError_t leg_fk_launch(LegKParams P, cudaStream_t st);
struct ServoKParams {
  int B, gait_mode;
  double half_hip_width, y_offset;
  const double *com, *theta, *rfoot, *lfoot;   // [3][B] each
  const double* homing;                         // [12][B], leg-major (FR, FL, RR, RL)
  double* q;                                    // [12][B] in/out: previous -> new joint angles
  double* jac;                                  // [36][B] or null
  double* foot_des;                             // [12][B] or null
  int* iters;                                   // [4][B] or null
};
cudaError_t servo_kin_launch(ServoKParams P, cudaStream_t st);
cudaError_t leg_ik_launch(LegKParams P, cudaStream_t st);
cudaError_t body_theta_gather_launch(int B, const double* body_out, int stride, double* theta, cudaStream_t st);
// device-resident body records (body_resident.cu)
cudaError_t body_record_expand_launch(int B, int nh, int in_stride, int tick_stride, int out_stride, const double* tx,
                                      const double* tick_in, const double* out_res, double* rec, int sms, cudaStream_t st);
cudaError_t body_record_pack_launch(int B, int nh, int out_stride, const double* out_res, double* tick_out, int sms, cudaStream_t st);

cudaError_t compact_pack_launch(int B, int nh, int out_stride, int diag_stride, const double* out38, const int* step_diag,
                                const double* body_out, const int* body_diag, double* compact, int sms, cudaStream_t st);

// ---- GRF distribution of the servo loop (grf_qp.cu) ----
constexpr int GRF_IN_DOUBLES = 48, GRF_OUT_DOUBLES = 16, GRF_DIAG_INTS = 32;
struct GrfKParams {
  int B, cap, warp_doubles;
  double qp_alpha, qp_beta, qp_gama, fz_max, mu;
  const double* in;     // [B][48]: base_p 3 | leg_p 12 (FR FL RR RL) | FT 6 | F_leg_guess 12 | grf_prev 12 | mode | right_support | pad
  double* out;          // [B][16]: grf 12 | cost | qp_solution | pad 2
  int* diag;            // [B][32] or null: status nactive iters[4] qp_solution 0 | active[24]
};
struct GrfDistParams {
  int B, mode;
  double y_coefficient;
  const double *com, *leg, *F, *rfoot, *lfoot;   // SoA [3][B], [12][B], [6][B], [3][B], [3][B]
  double* F_leg_ref;                             // SoA [12][B] (FR, FL, RR, RL xyz)
};
cudaError_t grf_force_opt_launch(GrfKParams P, int sms, cudaStream_t st);
int grf_warp_doubles();                          // shared-memory doubles of one force-QP warp: workspace | A | g0 | CE | ce0 | record
cudaError_t grf_force_distribution_launch(GrfDistParams P, cudaStream_t st);
struct GrfTauParams {
  int B;
  double swing_kp, swing_kd;
  const double* jac;                                   // [36][B], row-major 3x3 per leg (FR, FL, RR, RL)
  const int* swing;                                    // [4][B]
  const double *p_des, *p_est, *pv_des, *pv_est;       // [12][B]
  const double* F_leg_ref;                             // element k of robot b at [k * f_ks + b * f_bs]
  long long f_ks, f_bs;
  double* tau;                                         // [12][B]
};
cudaError_t grf_joint_torques_launch(GrfTauParams P, cudaStream_t st);

// ---- 40 Hz -> 100 Hz reference interpolation (ref_interp.cu) ----
struct RefInterpParams {
  int B, nh, t_end_footstep;
  double dt_sample;
  double inv[16];                 // _AAA_inv_mod, row-major
  const int* walktime;            // [B]
  const double* samples;          // [12][B]
  double* out;                    // [9 + 3 (nh - 1)][B]
};
cudaError_t ref_interp_launch(RefInterpParams P, cudaStream_t st);

// ---- signal filters of the servo loop (filters.cu) ----
constexpr int LPF_MAX_CHANNELS = 32;
struct LpfCoef { double b0, b1, b2, a1, a2, a; };
struct LpfKParams {
  int B, C;
  LpfCoef coef[LPF_MAX_CHANNELS];
  const double* in;        // [rows][B]: channel c reads row in_rows[c] (or row c when in_rows is null)
  const int* in_rows;      // device, [C] or null
  double* state;           // [5][C][B]
  double* out;             // [C][B]
};
cudaError_t lpf_launch(LpfKParams P, int sms, cudaStream_t st);
cudaError_t force_filter_launch(int B, int C, const double* in, double* state, double* out, int sms, cudaStream_t st);

// ---- the 40 Hz planner node (nlp_chain.cu): NLPRTControlClass around NLPClass; node state SoA [NLP_NODE_DOUBLES][B] ----
constexpr int NLP_NODE_DOUBLES = 480;
constexpr int NLP_NTD_MAX = 12;
struct NlpKParams {
  int B, walkdtime_max, t_end;
  double dt, dtx, height_offset_time, half_hip_width, stepwidth0, mass, rad, ggg, z_c, height_offset, Wn;
  double sh_w[NLP_NTD_MAX], ch_w[NLP_NTD_MAX];   // sinh / cosh(Wn dt jxx), jxx = 1..12: host libm
  const double* squat;        // [3][squat_n]: z, vz, az of X_CoM_position_squat at walktime = column (host table)
  int squat_n;
  double* node;               // [NLP_NODE_DOUBLES][B]
  const int* walkdtime;       // [B]
  const int* start;           // [B] or null (= 1)
  const int* cmd;             // [B] or null: 1 = StopWalking, 2 = StartWalking before this tick
  const double* rfoot_fb;     // [3][B] or null (= 0)
  const double* lfoot_fb;
  int* tick;                  // [B] workspace: the planner tick of the robot, 0 = no planner tick this call
  double* in;                 // [STEP_IN_DOUBLES][B] workspace: planner inputs
  double* out38;              // [38][B] workspace: planner outputs
  double* out18;              // [18][B] workspace: swing-foot outputs
  int* right_support;         // [B] workspace
  double* hz_co;              // [8][B] workspace
  double* lipm;               // [6][B] workspace
  double* msg;                // [100][B] /MPC/Gait
  const int* active;          // [B] or null (= every robot): robots with 0 skip the node -- no node row, tick input or message
                              //   slot is read or written, and their tick index is 0 so the planner kernels skip them too
};
cudaError_t nlp_pre_launch(NlpKParams P, cudaStream_t st);
cudaError_t nlp_post_launch(NlpKParams P, cudaStream_t st);

// ---- the 100 Hz node around the body MPC (rt_chain.cu): state SoA [field][B], messages SoA [100][B] ----
struct RtKParams {
  int B, nh, in_stride, out_stride;
  double dt_mpc, dt_slow, tstep, tdsp_ratio, stepwidth0, footx_max;
  double inv[16];                 // _AAA_inv_mod, row-major
  double* state;                  // [go1mpc_rt_node_state_doubles(nh)][B]
  const double* msg;              // [100][B] /MPC/Gait
  const int* ctrl;                // [B] control_gait(0) > 0, or null (= all on)
  const double* bodyangle_state;  // [4][B] or null (= 0)
  double* body_in;                // [B][in_stride] workspace: the body-MPC input records rt_pre_kernel assembles
  double* body_out;               // [B][out_stride] the body MPC's output records = its state
  double* out;                    // [100][B] /rtMPC/traj
  int* active;                    // [B] or null: 1 where the fast tick ran (message slot 99 > 0)
  // wire format of the node's other two topics (gait_fast.cpp:92-110, 519-527), optional: when ctl_msg is given it supplies the
  // control flag (slot 0) and the measured body angles (slots 10, 11, 13, 14) instead of ctrl / bodyangle_state
  const double* ctl_msg;          // [25][B] /control2rtmpc/state or null
  double* rt2nrt;                 // [25][B] /rt2nrt/state or null: slot 0 = t_int, slots 1..24 = the control message's
};
cudaError_t rt_pre_launch(RtKParams P, cudaStream_t st);
cudaError_t rt_post_launch(RtKParams P, cudaStream_t st);

// ---- the gait stack tick around both nodes (gait_stack.cu) ----
constexpr int GAIT_STACK_SENSOR_ROWS = 11, GAIT_STACK_SLOTS_MAX = 64;
struct GaitStackSlots {
  int n;
  int slot[GAIT_STACK_SLOTS_MAX];   // 0..99 /MPC/Gait slot, 100..199 /rtMPC/traj slot + 100
};
cudaError_t gait_stack_pre_launch(int B, int planner, double* walkdtime_row, int* walkdtime_i, const double* sensor, double* ctl,
                                  int sms, cudaStream_t st);
cudaError_t gait_stack_pack_launch(const GaitStackSlots& S, int B, const double* gait, const double* traj, double* rows, int sms,
                                   cudaStream_t st);
// per-robot clocks: plan[b] = whether robot b's planner ticks in this call (from clock[b], which is then incremented); walkdtime
// += 1 for those robots; the sensor scatter as gait_stack_pre_launch
cudaError_t gait_stack_clocked_pre_launch(int B, int* clock, int* plan, double* walkdtime_row, int* walkdtime_i, const double* sensor,
                                          double* ctl, int sms, cudaStream_t st);
// robot resets: ws = {count, 3 pad, flags[B], list[B]} ints, count zero on entry.  The mark kernel lists the flagged robots and does their
// small writes (clock 0, body record 0, servo rows); the column kernel writes the default column into the listed robots' state
struct StackResetParams {
  int B, rows, out_stride;
  const int* reset;           // [B]
  int* clock;                 // [B]
  double* state;              // [rows][B]
  const double* column;       // [rows] the default column
  double* body_out;           // [B][out_stride], 16-byte aligned
  double* servo;              // [SERVO_STATE_ROWS][B] or null
  double q0[12];              // servo joint angles after a reset
  int* count;
  int* list;                  // [B]
};
cudaError_t gait_stack_reset_launch(const StackResetParams& P, int sms, cudaStream_t st);
// farm health counters (farm_health.cu): int [FARM_HEALTH_ROWS][B] per farm, rows as GO1MPC_HEALTH_* of include/go1mpc.h
constexpr int FARM_HEALTH_ROWS = 12;
enum { FH_PLAN_OK = 0, FH_PLAN_INF = 1, FH_PLAN_FAIL = 2, FH_BODY_OK = 3, FH_BODY_INF = 4, FH_BODY_FAIL = 5, FH_GRF_OK = 6,
       FH_GRF_FAIL = 7, FH_GRF_FALLBACK = 8, FH_IK_CAP = 9, FH_NONFINITE = 10, FH_EVENTS = 11 };
// After a clocked gait stack tick: per robot, restart at clock 0 (clock after the call == 1), count the planner statuses of the
// robots whose node tick is >= 1, the body status, a non-finite rows_d row, and overwrite EVENTS
struct FarmHealthStackParams {
  int B, n_slots, body_diag_stride;
  const int* clock;           // [B] after the call
  const int* node_tick;       // [B] the planner node's tick index of this call (0: no planner tick)
  const int* step_diag;       // [STEP_DIAG_INTS][B]
  const int* body_diag;       // [B][body_diag_stride]
  const double* rows;         // [B][n_slots]
  int* health;                // [FARM_HEALTH_ROWS][B]
};
cudaError_t farm_health_stack_launch(const FarmHealthStackParams& P, int sms, cudaStream_t st);
// farm column copy: ws = {count, 3 pad, dst list[dst_B], src list[dst_B]} ints, count zero on entry.  The list kernel lists the
// destinations with a valid index and copies their clocks; the column kernel copies the listed columns' SoA rows (state | servo |
// force as one row range) and body records
struct FarmCopyParams {
  int dst_B, src_B;
  int rows, servo_end, soa_rows;    // state rows; + servo rows (0 or SERVO_STATE_ROWS); + force rows (0 or SERVO_FORCE_ROWS)
  int rec2;                         // double2 per body record
  const int* index;                 // [dst_B]
  int* bad;                         // or null
  double *dst_state, *dst_servo, *dst_force;
  const double *src_state, *src_servo, *src_force;
  double2* dst_body;
  const double2* src_body;
  int* dst_clock;                   // or null (then src_clock too)
  const int* src_clock;
  int* count;
  int *dlist, *slist;               // [dst_B]
  int* dst_health;                  // [FARM_HEALTH_ROWS][dst_B] or null (then src_health too): copied by the list kernel
  const int* src_health;            // [FARM_HEALTH_ROWS][src_B]
};
cudaError_t farm_copy_launch(const FarmCopyParams& P, int sms, cudaStream_t st);

// ---- the servo stack tick: K consecutive 1 kHz servo ticks from the gait stack's messages (servo_stack.cu) ----
constexpr int SERVO_TICKS_MAX = 10, SERVO_LPF_CHANNELS = 9;
constexpr int SERVO_ROW_Q = 0, SERVO_ROW_HOMING = 12, SERVO_ROW_LPF = 24, SERVO_STATE_ROWS = 24 + 5 * SERVO_LPF_CHANNELS;
struct ServoStackKParams {
  int B, K, gait_mode;
  double half_hip_width, y_offset;
  LpfCoef coef;                 // the 9 channels' filter (3 Hz at 1 kHz)
  const double* gait;           // [100][B] /MPC/Gait: slots 0 1 2 6 7 8 9 10 11 through the filters
  const double* traj;           // [100][B] /rtMPC/traj: slots 72, 73 = roll, pitch
  double* state;                // [SERVO_STATE_ROWS][B] in/out: q | homing | filters [5][9][B]
  double* q_out;                // [B][12 K] joint targets, tick-major per robot
  double* jac;                  // [36][B] or null (last tick)
  double* foot_des;             // [12][B] or null (last tick)
  int* iters;                   // [4][B] or null (last tick)
  double* ch;                   // [K][9][B] or null: each tick's filtered channels
  int* health;                  // [FARM_HEALTH_ROWS][B] or null: IK_CAP and EVENTS (servo_stack_kernel<true, true> only)
};
cudaError_t servo_stack_launch(const ServoStackKParams& P, cudaStream_t st);

// ---- the servo torque tick: force distribution, force QP and torque map after the servo stack (servo_torque.cu) ----
constexpr int SERVO_FORCE_ROWS = 24, SERVO_MEAS_ROWS = 24;
struct ServoTorqueKParams {
  GrfKParams g;                 // QP constants, cap and warp_doubles (in / out / diag unused)
  int B, K, gait_mode;
  double half_hip_width, y_offset, y_coefficient, swing_kp, swing_kd;
  const double* gait;           // [100][B] /MPC/Gait
  const double* traj;           // [100][B] /rtMPC/traj: slots 72, 73 = roll, pitch
  const double* homing;         // [12][B] the servo state's homing rows
  const double* ch;             // [K][9][B] filtered channels of each tick (servo_stack_kernel<true>)
  const double* q;              // [B][12 K] the IK's joint angles of each tick
  const double* meas;           // [24][B] measured q (12) and dq (12), FR FL RR RL
  const int* reset;             // [B] or null
  double* force;                // [SERVO_FORCE_ROWS][B] in/out: grf_opt 12 | F_leg_ref 12
  double* tau;                  // [B][12 K]
  double* grf;                  // [B][16] or null (last tick)
  int* grf_diag;                // [B][32] or null (last tick)
  int* health;                  // [FARM_HEALTH_ROWS][B] or null: force-QP rows, NONFINITE and EVENTS (servo_torque_kernel<4, true>)
};
cudaError_t servo_torque_launch(ServoTorqueKParams P, int sms, cudaStream_t st);

// register-resident DFMA loop: flops executed are returned through *flops
cudaError_t dfma_peak_launch(int grid, int block, int iters, double* sink, cudaStream_t st);

}  // namespace go1
