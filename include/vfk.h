/*
 * vfk.h -- C ABI of the batched vfclik control cycle for NVIDIA B200 (sm_100a).
 *
 * The reference (arcoslab/vfclik) has no FFI/plugin interface: its boundary is
 * process + YARP port + Python class.  This header is the boundary a maintainer
 * binds with ctypes (see INTEGRATION.md); each entry point names the reference
 * code it replaces.  Plain C types only; no exceptions cross the ABI; every call
 * returns VFK_OK (0) or a negative vfk_status and records a message retrievable
 * with vfk_last_error().
 *
 * One "control cycle" of one instance (SURVEY.md App. C.2) =
 *   FK + tool compose            scripts/vf:316-332         (Lafik/KDL FK)
 *   field evaluation + saturation scripts/vf:276-293,344-347 (vfl attractor / decay repellers)
 *   tool twist shift             scripts/vf:456-459         (PyKDL Twist.RefPoint)
 *   velocity IK                  scripts/vf:461             (Lafik.getIKV, weighted DLS)
 *   nullspace motion             scripts/nullspace:75-131,159-184
 *   joint P controller           scripts/joint_p_controller:79-89,126-146
 *   command mixer                src/command_mixer.py:71-82
 *   velocity clamp + command     scripts/bridge:188-203
 *   plant integration            (external joint_sim; explicit Euler)
 *
 * Data layout ("tile-blocked SoA"): instances are grouped in tiles of VFK_TILE = 32
 * (one warp).  A per-instance array with C components stores element (component c,
 * instance i) at
 *         base[ ((i / 32) * C + c) * 32 + i % 32 ]
 * The obstacle list {x, y, z, radius} is stored in PAIRS (obstacles 2p and 2p+1 of an
 * instance; an odd count M is padded with one zero-radius slot, Mp = M rounded up to
 * even), so that each lane's 16-byte vector holds the same component(s) of both
 * obstacles of a pair -- the operand form of sm_100's packed FP32 instructions, and a
 * conflict-free shared-memory access in both precisions.  With t = i / 32, l = i % 32,
 * p = m / 2, s = m % 2 and component c = 0..3 (x, y, z, radius), in scalars:
 *   precision 32:  base[ (((t * Mp/2 + p) * 2 + c/2) * 32 + l) * 4 + (c%2) * 2 + s ]
 *                  (two planes per pair: {x0, x1, y0, y1} and {z0, z1, r0, r1})
 *   precision 64:  base[ (((t * Mp/2 + p) * 4 + c) * 32 + l) * 2 + s ]
 *                  (four planes per pair: {x0, x1}, {y0, y1}, {z0, z1}, {r0, r1})
 * i.e. Mp * 32 * 4 scalars per tile either way.  obst_ext stores {safe distance, decay
 * order} of obstacle m of instance i at base[ ((t * M + m) * 32 + l) * 2 + k ].  A warp's
 * access to one component is one contiguous 128/256-byte line, and everything a warp
 * needs for a tile -- q, goal, each chunk of 8 obstacles -- is one contiguous burst moved
 * global -> shared by a single cp.async.bulk (TMA) copy.  Arrays cover
 * ceil(n_instances / 32) whole tiles (the padding lanes of the last tile must be
 * allocated; they are read, never written).  Base pointers must be 128-byte aligned.
 * Element type is float (precision 32) or double (precision 64) as chosen at
 * vfk_create().  vfk_pack()/vfk_unpack() convert dense SoA [C][n] device arrays to and
 * from this layout; the host-buffer session API takes plain dense arrays.
 */
#ifndef VFK_H_
#define VFK_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* 0.1.0.  vfk_buffers grew by the mixed-scene fields at its end (VFK_OBST_MIXED) without a new version: the library
 * reads them only when obst_shared == VFK_OBST_MIXED, which no caller built against the shorter struct can set, and
 * vfk_session_buffers writes them only for a session switched to that mode, so an older caller's struct is never read
 * or written past its end. */
#define VFK_VERSION 100
#define VFK_MAX_JOINTS 17
#define VFK_TILE 32              /* instances per layout tile */
#define VFK_N_PORTS 6            /* mixer inputs, order of scripts/bridge:593-596 */
#define VFK_GOAL_COMPS 13        /* R_goal row-major (9), p_goal (3), slowdown distance (1) */
#define VFK_POSE_COMPS 12        /* R row-major (9), p (3) */
#define VFK_AUX_COMPS 12         /* auxiliary field record: type, force, 10 parameters */
#define VFK_MAX_SHARED_OBSTACLES 1024  /* largest shared obstacle list (vfk_buffers.obst_shared = 1 or 2) */

/* vfk_buffers.obst_shared: which obstacle lists a call uses */
enum { VFK_OBST_PER_INSTANCE = 0,  /* obst / obst_ext per instance (blocked layout above) */
       VFK_OBST_SHARED = 1,        /* obst / obst_ext: one dense list for the whole batch */
       VFK_OBST_MIXED = 2 };       /* obst / obst_ext per instance (n_obstacles of them) plus shared_obst / shared_obst_ext,
                                      one dense list of n_shared_obst for the whole batch */

typedef enum vfk_status {
    VFK_OK = 0,
    VFK_ERR_INVALID = -1,        /* bad argument (message says which) */
    VFK_ERR_UNSUPPORTED = -2,    /* e.g. n_joints without a compiled kernel, control mode with N != 7 */
    VFK_ERR_CUDA = -3,           /* a CUDA runtime call failed */
    VFK_ERR_NO_DEVICE = -4       /* no sm_100 device: there is no CPU fallback */
} vfk_status;

/* KDL joint types (PyKDL Joint.*); fixed segments are folded on the host. */
enum { VFK_JOINT_NONE = 0, VFK_JOINT_ROTX, VFK_JOINT_ROTY, VFK_JOINT_ROTZ,
       VFK_JOINT_TRANSX, VFK_JOINT_TRANSY, VFK_JOINT_TRANSZ };

/* per-instance flag bits written to vfk_buffers.flags */
enum { VFK_FLAG_AT_GOAL = 1,     /* scripts/joint_p_controller:135-146 (signed compare, no abs) */
       VFK_FLAG_NS_LIMIT = 2,    /* scripts/nullspace:120-131 zeroed the nullspace command */
       VFK_FLAG_NAN = 4,         /* src/command_mixer.py:71-75 */
       VFK_FLAG_CLAMPED = 8 };   /* scripts/bridge:190-196 ratio < 1 */

enum { VFK_NS_OFF = 0,           /* --no_nullspace (scripts/vfclik:73-79) */
       VFK_NS_PROJECTOR = 1,     /* qdot_ns = gain * check((I - J^+ J) qdot0) */
       VFK_NS_CONTROL = 2 };     /* the reference's 4-float control interface (scripts/nullspace:110-117): qdot_ns =
                                    gain * check(sum_{i < min(4, k)} control_i u_i), u_i an orthonormal basis of null(J),
                                    k = N - 6 vectors, each kept sign-continuous from cycle to cycle.  Any N; ns_lambda unused. */

/* Velocity IK behind Lafik.getIKV (scripts/vf:461).  The solver itself is un-vendored (KDL through arcospyu):
 *   DLS        north_star's form, qdot = Wj Jw^T (Jw Jw^T + lambda^2 I)^-1 Wt t -- every singular value damped; both precisions
 *   TRUNCATED  qdot = Wj V diag(f(sigma)) U^T Wt t with f = 1 / sigma for sigma >= ik_eps and sigma / (sigma^2 + lambda^2) below
 *              -- how KDL's ChainIkSolverVel_wdls is recalled to treat lambda (a plain weighted pseudo-inverse away from
 *              singularities); one-sided Jacobi SVD of Jw in the kernel, precision 64 only.  Provided so that a comparison
 *              against a real Lafik, should one become available, is one flag away. */
enum { VFK_IK_DLS = 0, VFK_IK_TRUNCATED = 1 };

/* Robot back-end whose set_vel() the clamp / command step restates (SURVEY.md section 8 row f4):
 *   LWR       leading-joint clamp; cmd = qdot_lim (direct) or -q_cmded + q + qdot_lim      (scripts/bridge:182-210)
 *   POWERCUBE leading-joint clamp, then the shoulder-speed clamp of joint 0.  Bug-compatible: the reference reuses one
 *             `ratio` variable, so when the shoulder limit is NOT hit the leading ratio is applied a second time
 *             (scripts/bridge:288-305); cmd = qdot_lim
 *   ICUB      leading-joint clamp; cmd = qdot_lim (scripts/bridge:507-530; inactive torso joints are handled through the
 *             joint weights the bridge sends to the vector field, :470-500) */
enum { VFK_BRIDGE_LWR = 0, VFK_BRIDGE_POWERCUBE = 1, VFK_BRIDGE_ICUB = 2 };

/* Serial chain: flange = base * prod_i ( Joint_i(q_i) * tip_i ).  Frames are 12
 * doubles: R row-major (9) then p (3).  Replaces the PyKDL chain Lafik builds from
 * config.segments (scripts/vf:153). */
typedef struct vfk_chain_desc {
    int32_t n_joints;
    int32_t joint_type[VFK_MAX_JOINTS];
    double base[12];
    double tip[VFK_MAX_JOINTS][12];
    double q_lo[VFK_MAX_JOINTS];
    double q_hi[VFK_MAX_JOINTS];
} vfk_chain_desc;

/* Per-robot constants (uniform over the batch; kept in constant memory). */
typedef struct vfk_params {
    double ik_lambda;            /* damping of J^T (J J^T + lambda^2 I)^-1           (getIKV, scripts/vf:461) */
    double ns_lambda;            /* damping of the projector's pseudo-inverse (VFK_NS_PROJECTOR); 0 = the reference's
                                    I - pinv(J) J (scripts/nullspace:78), computed through a one-sided Jacobi SVD of J with
                                    pinv's cutoff, so it projects onto all of null(J) where J loses rank (error cond(J)*eps;
                                    FP32 cuts singular values below 1e-6 sigma_max, see vfk_nullspace.cuh).  FP32 mode needs ik_lambda > 0: the undamped normal equations
                                    of the velocity IK lose their pivots to FP32 rounding near singular postures */
    double dt;                   /* config.rate (scripts/bridge:91) */
    double speed_scale;          /* speedScale (scripts/vf:137,197-207) */
    double max_vel;              /* scripts/bridge:69,613-623 */
    double jp_kp;                /* config.jpctrl_kp (scripts/joint_p_controller:56) */
    double jp_delta;             /* 0.087 (scripts/joint_p_controller:57) */
    double ns_gain;              /* 0.5 (scripts/nullspace:62,183) */
    double ns_lookahead;         /* 0.3 (scripts/nullspace:121) */
    double ns_limit_gain;        /* k of qdot0_i = -k (q_i - mid_i)/(hi_i - lo_i)^2 */
    double rot_slowdown;         /* angle below which the rotational speed ramps down */
    double goal_force;           /* +1  (scripts/object_feeder:236) */
    double obst_force;           /* -10 (scripts/object_feeder:322) */
    double obst_safe;            /* 0.001 (scripts/object_feeder:331), used when vfk_buffers.obst_ext == NULL */
    double obst_order;           /* decay order (> 0), used when vfk_buffers.obst_ext == NULL */
    double mixer_w[VFK_N_PORTS]; /* [vectorfield, nullspace, joint, mechanism, xtra1, xtra2] */
    double w_task[6];            /* diag of set_tweights (scripts/vf:296-305) */
    double w_joint[VFK_MAX_JOINTS]; /* diag of set_jweights (scripts/vf:306-309) */
    double tool[12];             /* tool frame in the flange frame (scripts/vf:321-330) */
    double jp_ref[VFK_MAX_JOINTS];  /* used when vfk_buffers.jp_ref == NULL (config.initial_joint_pos) */
    double ns_control[4];        /* used in VFK_NS_CONTROL when vfk_buffers.ns_in == NULL */
    double shoulder_vel[2];      /* VFK_BRIDGE_POWERCUBE: config.max_vel_shoulder_pos (> 0), max_vel_shoulder_neg (< 0)
                                    (scripts/bridge:296-303) */
    double ik_eps;               /* VFK_IK_TRUNCATED: singular values below this are damped, the rest inverted plainly */
    int32_t ns_mode;             /* VFK_NS_* */
    int32_t direct_control;      /* -1: auto = all mixer weights zero (scripts/bridge:604); 0 / 1 force */
    int32_t integrate;           /* 1: q += dt * qdot_lim after every cycle (simulation plant) */
    int32_t bridge_kind;         /* VFK_BRIDGE_*: which set_vel the clamp / command step follows */
    int32_t ik_mode;             /* VFK_IK_*: form of the velocity IK (scripts/vf:461, Lafik.getIKV) */
    int32_t reserved;
} vfk_params;

/* Device buffers of one vfk_step() call, all in the tile-blocked layout above
 * ("[C]" = C components per instance).  NULL = not supplied / not wanted. */
typedef struct vfk_buffers {
    void*       q;               /* [N]  in; out when params.integrate                            */
    const void* goal;            /* [13] attractor (vfl type 1) per instance                       */
    const void* obst;            /* M obstacles x {x, y, z, radius}, pair-interleaved (see above): decay repellers (vfl type 2);
                                    radius 0 = empty slot (the padding slot of an odd M must be zero) */
    const void* obst_ext;        /* M obstacles x {safe distance, decay order} (wire-faithful,
                                    scripts/object_feeder:326-333) or NULL -> params.obst_safe / obst_order */
    const void* aux;             /* [n_aux * 12] auxiliary field records {type, force, p0..p9} or NULL:
                                    type 4 hemisphere repeller {x,y,z, nx,ny,nz, safe, order} (scripts/object_feeder:335-354),
                                    type 5 funnel attractor {x,y,z, ax,ay,az, cut angle, angle order, cut distance, distance order}
                                    (scripts/object_feeder:262-280); other type codes = empty slot */
    void*       jp_ref;          /* [N]  joint reference (/jpctrl/ref) or NULL -> params.jp_ref.  In/out when jp_lo / jp_hi are
                                    given: the clamped reference is stored back, like the `ref` variable of the reference's loop
                                    (scripts/joint_p_controller:121), so a clamp persists when the limits later widen */
    const void* ns_in;           /* PROJECTOR: qdot0 [N] or NULL -> limit-avoidance gradient;
                                    CONTROL:   control [4] or NULL -> params.ns_control             */
    void*       ns_lastvec;      /* CONTROL: [min(4, N-6) * N] in/out: the basis vectors of the previous cycle, vector i at
                                    components i*N .. i*N+N-1 -- the sign-continuity state `lastvec` of scripts/nullspace:91-107
                                    (start zeroed).  Not needed when N <= 6 (empty nullspace). */
    const void* q_cmded;         /* [N]  last commanded q (scripts/bridge:169-172) or NULL -> q     */
    const void* ext_cmd[3];      /* mixer ports 3..5, [N] each, or NULL -> 0                        */
    void*       qdot_vf;         /* out [N]  /vectorField/qdotOut                                  */
    void*       qdot_ns;         /* out [N]  /nullspace/qdotout                                    */
    void*       qdot_jp;         /* out [N]  /jpctrl/out                                           */
    void*       qdot;            /* out [N]  clamped mixer output qdot_lim (scripts/bridge:196)    */
    void*       cmd;             /* out [N]  command sent to the plant (scripts/bridge:198-203)    */
    void*       pose;            /* out [12] tool frame (/vectorField/pose)                        */
    void*       twist;           /* out [6]  commanded tool twist velPos, velRot (/vectorField/vector_out, scripts/vf:346-347) */
    int32_t*    flags;           /* out [1]  VFK_FLAG_*                                            */
    int32_t     n_aux;           /* slots in aux (0..64)                                           */
    int32_t     obst_shared;     /* VFK_OBST_*.  0: obst / obst_ext are per instance (layout above).  1: one scene for the
                                    whole batch: obst is dense [M][4] {x, y, z, radius} and obst_ext (or NULL) dense [M][2]
                                    {safe, order}, in the handle's precision, 128-byte aligned, M <= VFK_MAX_SHARED_OBSTACLES
                                    (larger M: VFK_ERR_UNSUPPORTED).  Each CTA reads the list into shared memory once per
                                    launch, so an instance costs no obstacle traffic at all; the field is bit-identical to the
                                    per-instance path given the same list replicated to every instance.  2: both -- obst /
                                    obst_ext per instance as in mode 0 (n_obstacles = Mi of them) and the shared list in
                                    shared_obst / shared_obst_ext below; see those fields.  aux stays per instance.  This field
                                    was once reserved: C callers must zero it (ctypes structures start zeroed).  A library
                                    that has it exports vfk_session_set_shared_obstacles (modes 0 / 1) and
                                    vfk_session_use_obstacles (mode 2). */
    const void* jp_lo;           /* [N]  per-instance joint limits the joint controller clamps its reference into --      */
    const void* jp_hi;           /* [N]  config.updateJntLimits(q) (scripts/joint_p_controller:79-89; posture-dependent on the
                                    iCub) evaluated by the caller per instance -- or NULL (both) -> the chain's static limits */
    /* Read only when obst_shared == VFK_OBST_MIXED (appended fields: a caller built against the struct without them never
     * sets that mode).  The field of an instance sums its own Mi obstacles first, then the Ms shared ones, as if its list
     * were [own ; shared]; it equals mode 0 on that concatenated list bit for bit when Mi is a multiple of 8 (the repulsor
     * works in chunks of 8) and to rounding otherwise.  Ms = 0 runs exactly the per-instance call, Mi = 0 exactly mode 1. */
    const void* shared_obst;     /* dense [Ms][4] {x, y, z, radius}, 128-byte aligned; required in this mode even when Ms = 0
                                    (a mode-2 call without it is refused rather than read a shared-only obst as per instance) */
    const void* shared_obst_ext; /* dense [Ms][2] {safe, order}, 128-byte aligned, or NULL.  With both lists non-empty, obst_ext
                                    and shared_obst_ext come both or neither (VFK_ERR_INVALID otherwise) */
    int32_t     n_shared_obst;   /* Ms in 0..VFK_MAX_SHARED_OBSTACLES (< 0: VFK_ERR_INVALID; larger: VFK_ERR_UNSUPPORTED) */
    int32_t     reserved2;       /* must be 0 */
} vfk_buffers;

typedef struct vfk_ctx* vfk_handle;
typedef struct vfk_session_s* vfk_session;

int  vfk_version(void);
void vfk_default_params(vfk_params* out, int n_joints);

/* precision: 32 or 64.  device: CUDA ordinal.  Fails with VFK_ERR_NO_DEVICE when
 * the device is not compute capability 10.x (no fallback path exists). */
int  vfk_create(vfk_handle* out, const vfk_chain_desc* chain, int precision, int device);
int  vfk_set_params(vfk_handle h, const vfk_params* p);
int  vfk_get_params(vfk_handle h, vfk_params* out);
/* Which compile-time chain pattern the handle's kernels use: 0 = generic (any chain),
 * 1 = LWR-style 7R structure (tip rotations are +-90 degree twists, sparse offsets),
 * 2 = Denavit-Hartenberg form (10 or 17 revolute joints, every tip rotation RotX(alpha)). */
int  vfk_chain_pattern(vfk_handle h);
void vfk_destroy(vfk_handle h);
const char* vfk_last_error(vfk_handle h);   /* h may be NULL: last error of vfk_create */

/* K fused control cycles over n_instances instances, stream-ordered on `stream`
 * (a cudaStream_t, may be NULL).  No allocation, no synchronisation.
 * Outputs hold the last cycle's values.  Returns the number of kernels launched
 * (>= 1) or a negative vfk_status. */
int  vfk_step(vfk_handle h, const vfk_buffers* bufs, int64_t n_instances, int n_obstacles,
              int k_cycles, void* stream);

/* Run each instance's control loop until its tool reaches the goal: the batched HandleArm.gotoFrame / gotThere
 * (src/handlers.py:346-387), which poll the distance monitor until the tool is within goal_precision.  Inputs and
 * parameters as for vfk_step (params.integrate must be 1).  q_c = q after c cycles; the rule at q_c is
 *     |p_goal - p_tool| < tol_trans (metres)  and  angle(R_goal R_tool^T) < tol_rot (radians, [0, pi])
 * for the tool frame (params.tool), strict as in the reference; tol_rot >= pi drops the orientation condition, and a
 * tolerance of 0 can never be met.  Per instance:
 *     cycles_out [1] (int32, blocked)  the smallest c in 0..max_cycles with the rule at q_c, or -1 if there is none;
 *     q (in/out)                       q_c for that c (the instance stops there: no further integration), else q_max_cycles;
 *     dist_out [2] (blocked, or NULL)  {|p_goal - p_tool|, angle} at the returned q;
 *     jp_ref (with jp_lo / jp_hi) and ns_lastvec hold the state of the instance's last cycle, as after vfk_step.
 * The returned q is bit-identical to vfk_step with k_cycles = cycles_out (or max_cycles) on the same batch.  A warp
 * whose 32 instances have all stopped takes its next tile, so converged work costs nothing.  The per-cycle outputs of
 * vfk_buffers (qdot_vf, qdot_ns, qdot_jp, qdot, cmd, pose, twist, flags) must be NULL: they have no single meaning in
 * a batch whose instances stop at different cycles.  In precision 32 the tool frame is rounded to float (6e-8), so
 * tolerances below about 1e-6 m / 1e-6 rad may never be met.  No allocation, no synchronisation; returns the number
 * of kernels launched or a negative vfk_status. */
int  vfk_solve(vfk_handle h, const vfk_buffers* bufs, int64_t n_instances, int n_obstacles, int max_cycles,
               double tol_trans, double tol_rot, int32_t* cycles_out, void* dist_out, void* stream);

/* Field visualisation query (scripts/vf:469-503): twist the composed field commands at
 * arbitrary tool poses pose_in [12]; twist_out [6] (blocked layout).  Same goal/obst layout. */
int  vfk_field_eval(vfk_handle h, const void* pose_in, const void* goal, const void* obst,
                    const void* obst_ext, const void* aux, int n_aux, void* twist_out,
                    int64_t n_instances, int n_obstacles, void* stream);
/* The same query on the scene a vfk_step call would use: goal, obst, obst_ext, aux, n_aux, obst_shared and, in
 * VFK_OBST_MIXED, the shared_* fields are taken from `scene` (every other field is ignored); n_obstacles means what it
 * means to vfk_step (mode 1: the shared list's length; mode 2: the per-instance count).  Sums the own obstacles, then
 * the shared ones, one at a time: bit-identical to vfk_field_eval on the replicated or concatenated per-instance list. */
int  vfk_field_eval_scene(vfk_handle h, const void* pose_in, const vfk_buffers* scene, int64_t n_instances, int n_obstacles,
                          void* twist_out, void* stream);

/* Weighted sum of command ports (src/command_mixer.py:78-82) on device buffers:
 * out(c, i) = sum_p w[p] * cmds[p](c, i); cmds[p] may be NULL (skipped); nan_flags [1] optional. */
int  vfk_mix(vfk_handle h, const void* const* cmds, const double* w, int n_ports, int n_channels,
             void* out, int32_t* nan_flags, int64_t n_instances, void* stream);

/* LWR_Bridge.set_vel (scripts/bridge:188-203) on device buffers [n_channels]: ratio = max_vel / max_c |qdot_c| when
 * exceeded; cmd = qdot_lim if direct_control else -q_cmded + q + qdot_lim (q_cmded NULL -> q). qdot_lim_out optional.
 * params.bridge_kind selects the back-end: VFK_BRIDGE_POWERCUBE adds the shoulder clamp of Powercube_Bridge.set_vel
 * (scripts/bridge:288-305), and it and VFK_BRIDGE_ICUB (:507-530) always command qdot_lim itself. */
int  vfk_set_vel(vfk_handle h, const void* qdot, const void* q, const void* q_cmded, double max_vel, int direct_control,
                 void* cmd_out, void* qdot_lim_out, int n_channels, int64_t n_instances, void* stream);

/* Monitoring (SURVEY.md section 8 row f1), one call per control cycle after vfk_step:
 *   tracking-error diagnostics of scripts/vf:349-428 -> track_out [8] (the 7 doubles + arm_tracking of /vectorField/track_error),
 *   distance monitor of scripts/monitor_distance:76-84,148-219 -> dist_out [2] (metres, degrees to the goal) and
 *   tracking_state_out [2] int32 (majority over the last 20 cycles: 0 on goal, 1 follow, 2 not follow; -1 before 21 samples).
 * pose [12] and twist [6] are vfk_step outputs; state_f [32] and state_i [6] (int32) carry the 5-frame / 4-command
 * history between calls and must start zeroed.  Outputs may be NULL. */
int  vfk_monitor(vfk_handle h, const void* pose, const void* twist, const void* goal, void* state_f, int32_t* state_i,
                 void* track_out, void* dist_out, int32_t* tracking_state_out, int64_t n_instances, void* stream);

/* Layout conversion on the device: dense SoA [comps][n] (width scalars per element: 1 for
 * per-instance components, 2 for obst_ext [M][n][2]) <-> tile-blocked; width 4 = the obstacle list:
 * dense [M][n][4] <-> the pair-interleaved blocked array (Mp rows per tile, padding slot zeroed). */
int  vfk_pack(vfk_handle h, const void* dense, void* blocked, int comps, int width, int64_t n_instances, void* stream);
int  vfk_unpack(vfk_handle h, const void* blocked, void* dense, int comps, int width, int64_t n_instances, void* stream);

/* ---- host-buffer sessions: the call a host-language plugin makes --------------
 * A session owns resident device copies of the scene (goal, obstacles) and state,
 * pinned staging buffers and a stream.  Host arrays are plain dense SoA of the handle's
 * precision: [comps][n_instances] (obstacles [M][n][4], ext [M][n][2]); the session
 * converts to / from the blocked layout on the GPU.  vfk_session_cycle()
 * takes q from the host (if q_in != NULL), runs k_cycles fused cycles, returns the
 * requested outputs to the host and synchronises.  How the data moves depends on the
 * caller's buffers, never on the results (bit-identical either way):
 *   - q_in (and qdot_out, if wanted) page-locked -- cudaHostAlloc, cudaHostRegister,
 *     torch pin_memory() -- 16-byte aligned, n_instances a multiple of 32 and >= 1024:
 *     ONE launch of the cycle kernel reads the q tiles from and writes qdot to the host
 *     buffers itself over PCIe (no staging copies, no layout kernels);
 *   - otherwise: a chunked copy pipeline (H2D / pack / cycle / unpack / D2H on three
 *     streams), pageable buffers going through the session's pinned staging area. */
int  vfk_session_create(vfk_handle h, int64_t n_instances, int n_obstacles, int with_obst_ext, vfk_session* out);
int  vfk_session_set_goal(vfk_session s, const void* goal_host);            /* [13][n] */
int  vfk_session_set_obstacles(vfk_session s, const void* obst_host,         /* [M][n][4] */
                               const void* obst_ext_host);                  /* [M][n][2] or NULL */
/* One scene for every instance (vfk_buffers.obst_shared): copies obst_host [M][4] and obst_ext_host [M][2] (or NULL ->
 * params.obst_safe / obst_order) to a device buffer the session owns, M in 0..VFK_MAX_SHARED_OBSTACLES.  From then on
 * vfk_session_cycle, vfk_session_solve and vfk_session_buffers use it, until vfk_session_set_obstacles is called on a
 * session created with n_obstacles > 0 (on one created with 0 that call stays a no-op).  A session created with
 * n_obstacles = 0 allocates no per-instance scene. */
int  vfk_session_set_shared_obstacles(vfk_session s, const void* obst_host, const void* obst_ext_host, int n_obstacles);
/* Which lists vfk_session_cycle, vfk_session_solve and vfk_session_buffers use: VFK_OBST_PER_INSTANCE,
 * VFK_OBST_SHARED (needs a shared list) or VFK_OBST_MIXED (needs a session created with n_obstacles > 0 and a shared list;
 * when both are non-empty their ext rows come both or neither).  Otherwise VFK_ERR_INVALID.  The two setters above
 * keep their side effects (set_obstacles selects mode 0, set_shared_obstacles mode 1): call this after both. */
int  vfk_session_use_obstacles(vfk_session s, int mode);
int  vfk_session_set_aux(vfk_session s, const void* aux_host, int n_aux);   /* [n_aux * 12][n] records, or NULL / 0 to clear */
int  vfk_session_set_q(vfk_session s, const void* q_host);                  /* [N][n] */
int  vfk_session_set_jp_ref(vfk_session s, const void* ref_host);           /* [N][n] or NULL -> params.jp_ref */
int  vfk_session_set_jp_limits(vfk_session s, const void* lo_host,          /* [N][n] each: per-instance limits of the joint */
                               const void* hi_host);                        /* controller, or NULL (both) -> the chain's */
int  vfk_session_set_ns_input(vfk_session s, const void* ns_host);          /* [N|4][n] or NULL */
int  vfk_session_cycle(vfk_session s, const void* q_in_host, int k_cycles,
                       void* qdot_out_host, void* q_out_host, int32_t* flags_out_host);
/* vfk_solve on the session's resident scene and state: q from the host (if q_in != NULL, through vfk_session_set_q),
 * the stop rule as in vfk_solve, then q_out [N][n], cycles_out [n] (int32) and dist_out [2][n] back to the host (each
 * may be NULL); synchronises. */
int  vfk_session_solve(vfk_session s, const void* q_in_host, int max_cycles, double tol_trans, double tol_rot,
                       void* q_out_host, int32_t* cycles_out_host, void* dist_out_host);
/* Optional per-controller outputs the kernel writes each cycle ("qdot_vf","qdot_ns","qdot_jp","cmd","pose","twist");
 * all off by default so the resident path only moves q in and qdot out. */
int  vfk_session_enable(vfk_session s, const char* what, int on);
int  vfk_session_read(vfk_session s, const char* what, void* out_host);     /* enabled outputs, "qdot", "q", "lastvec" */
int  vfk_session_buffers(vfk_session s, vfk_buffers* out);                  /* blocked device view (stream-ordered use) */
void vfk_session_destroy(vfk_session s);

#ifdef __cplusplus
}
#endif
#endif /* VFK_H_ */
