// vfk_api.cu -- C ABI (include/vfk.h) over the fused control-cycle kernel.
//
// Host side only prepares constants and launches; there is no CPU compute path:
// vfk_create() fails with VFK_ERR_NO_DEVICE when no sm_100 GPU is present.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <new>

#include "vfk_ctx.cuh"

using namespace vfk;

// -------------------------------------------------------------------------------- frames (host, double)
static void frame_mul(const double* a, const double* b, double* o) {
    double r[12];
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j)
            r[3 * i + j] = a[3 * i] * b[j] + a[3 * i + 1] * b[3 + j] + a[3 * i + 2] * b[6 + j];
        r[9 + i] = a[3 * i] * b[9] + a[3 * i + 1] * b[10] + a[3 * i + 2] * b[11] + a[9 + i];
    }
    memcpy(o, r, sizeof r);
}

// RotX/RotY/TransX/TransY joints are conjugated into Z joints:  Joint_axis(q) = C JointZ(q) C^T
// with C e_z = e_axis.  C is appended to the frame before the joint and C^T prepended to its tip,
// so the kernel only ever rotates about / translates along the local Z axis.
static void canonicalise_chain(const vfk_chain_desc& in, vfk_chain_desc& out) {
    out = in;
    static const double CX[12] = {0, 0, 1, 0, 1, 0, -1, 0, 0, 0, 0, 0};    // RotY(+pi/2): z -> x
    static const double CXt[12] = {0, 0, -1, 0, 1, 0, 1, 0, 0, 0, 0, 0};
    static const double CY[12] = {1, 0, 0, 0, 0, 1, 0, -1, 0, 0, 0, 0};    // RotX(-pi/2): z -> y
    static const double CYt[12] = {1, 0, 0, 0, 0, -1, 0, 1, 0, 0, 0, 0};
    for (int j = 0; j < in.n_joints; ++j) {
        const int t = in.joint_type[j];
        const double *C = nullptr, *Ct = nullptr;
        if (t == VFK_JOINT_ROTX || t == VFK_JOINT_TRANSX) { C = CX; Ct = CXt; }
        if (t == VFK_JOINT_ROTY || t == VFK_JOINT_TRANSY) { C = CY; Ct = CYt; }
        if (C) {
            double* prev = (j == 0) ? out.base : out.tip[j - 1];
            frame_mul(prev, C, prev);
            frame_mul(Ct, out.tip[j], out.tip[j]);
        }
        out.joint_type[j] = (t >= VFK_JOINT_TRANSX) ? VFK_JOINT_TRANSZ : VFK_JOINT_ROTZ;
    }
}

// Does the canonical chain have the structure PAT assumes (tip rotations = the pattern's signed
// permutations, tip translations zero where the pattern drops them, identity base rotation)?
template <class PAT>
static bool chain_matches(const vfk_chain_desc& ch, int n_expected) {
    if (ch.n_joints != n_expected) return false;
    static const double ident[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    if (PAT::base_identity && memcmp(ch.base, ident, sizeof ident) != 0) return false;
    for (int j = 0; j < ch.n_joints; ++j) {
        if (ch.joint_type[j] != VFK_JOINT_ROTZ) return false;
        for (int k = 0; k < 3; ++k) {
            for (int r = 0; r < 3; ++r) {            // column k of R_tip = sign * e_perm
                const double want = (r == PAT::perm(j, k)) ? (double)PAT::sign(j, k) : 0.0;
                if (ch.tip[j][3 * r + k] != want) return false;
            }
            if (!PAT::pnz(j, k) && ch.tip[j][9 + k] != 0.0) return false;
        }
    }
    return true;
}

template <typename T>
static void build_const(const vfk_ctx& h, KConst<T>& c) {
    memset(&c, 0, sizeof c);
    c.sincos = sincos_tab();
    const vfk_chain_desc& ch = h.canon;
    const vfk_params& p = h.params;
    const int n = ch.n_joints;
    for (int k = 0; k < 12; ++k) c.base[k] = ch.base[k];
    bool unit = true, all_xt = true;
    for (int j = 0; j < n; ++j) {
        for (int k = 0; k < 12; ++k) c.tip[j][k] = ch.tip[j][k];
        c.q_lo[j] = (T)ch.q_lo[j];
        c.q_hi[j] = (T)ch.q_hi[j];
        const double rng = ch.q_hi[j] - ch.q_lo[j];
        c.ns_q0_scale[j] = (T)(-p.ns_limit_gain / (rng * rng));
        c.ns_mid[j] = (T)(0.5 * (ch.q_lo[j] + ch.q_hi[j]));
        c.w_joint[j] = (T)p.w_joint[j];
        c.jp_ref[j] = (T)p.jp_ref[j];
        if (p.w_joint[j] != 1.0) unit = false;
        if (ch.joint_type[j] == VFK_JOINT_TRANSZ) c.prismatic_mask |= (1 << j);
        // structure of the tip rotation (exact tests: the fast paths must give the general product's value)
        const double* r = ch.tip[j];
        const bool xtwist = r[0] == 1.0 && r[1] == 0.0 && r[2] == 0.0 && r[3] == 0.0 && r[6] == 0.0 && r[4] == r[8] && r[5] == -r[7];
        if (xtwist && r[4] == 1.0 && r[7] == 0.0) c.tipident_mask |= (1 << j);
        else if (xtwist) c.xtwist_mask |= (1 << j);
        if (!xtwist) all_xt = false;
    }
    c.all_xtwist = all_xt ? 1 : 0;
    bool all_zero = true;
    for (int k = 0; k < 6; ++k) {
        c.w_task[k] = (T)p.w_task[k];
        c.mixer_w[k] = (T)p.mixer_w[k];
        if (p.w_task[k] != 1.0) unit = false;
        if (p.mixer_w[k] != 0.0) all_zero = false;
    }
    static const double ident[12] = {1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0};
    c.tool_identity = memcmp(p.tool, ident, sizeof ident) == 0;
    for (int k = 0; k < 12; ++k) c.tool[k] = (T)p.tool[k];
    for (int k = 0; k < 4; ++k) c.ns_control[k] = (T)p.ns_control[k];
    c.ik_lambda2 = (T)(p.ik_lambda * p.ik_lambda);
    c.ns_lambda2 = (T)(p.ns_lambda * p.ns_lambda);
    c.dt = (T)p.dt;
    c.speed_scale = (T)p.speed_scale;
    c.max_vel = (T)p.max_vel;
    c.jp_kp = (T)p.jp_kp;
    c.jp_delta = (T)p.jp_delta;
    c.ns_gain = (T)p.ns_gain;
    c.ns_lookahead = (T)p.ns_lookahead;
    c.rot_slowdown_inv = (T)(p.rot_slowdown > 0 ? 1.0 / p.rot_slowdown : INFINITY);
    c.goal_force = (T)p.goal_force;
    c.obst_force = (T)p.obst_force;
    c.obst_safe_inv = (T)(p.obst_safe > 0 ? 1.0 / p.obst_safe : INFINITY);
    c.obst_order = (T)p.obst_order;
    c.ns_mode = p.ns_mode;
    c.direct_control = p.direct_control < 0 ? (all_zero ? 1 : 0) : (p.direct_control ? 1 : 0);
    if (p.bridge_kind != VFK_BRIDGE_LWR) c.direct_control = 1;          // Powercube / iCub command qdot_lim itself
    c.shoulder_clamp = p.bridge_kind == VFK_BRIDGE_POWERCUBE;
    c.shoulder_pos = (T)p.shoulder_vel[0];
    c.shoulder_neg = (T)p.shoulder_vel[1];
    c.integrate = p.integrate ? 1 : 0;
    c.unit_weights = unit ? 1 : 0;
    // the reference's nullspace (control interface: Householder basis of null(J)) and the undamped projector (one-sided
    // Jacobi SVD of J, rank-revealing) skip the normal equations (vfk_nullspace.cuh): no cond(J)^2, no pivot to lose at
    // ns_lambda = 0
    c.ns_qr = (p.ns_mode == VFK_NS_CONTROL || (p.ns_mode == VFK_NS_PROJECTOR && p.ns_lambda == 0.0)) ? 1 : 0;
    c.share_factor = (unit && p.ns_lambda == p.ik_lambda && !c.ns_qr) ? 1 : 0;
    c.ik_mode = p.ik_mode;
    c.ik_eps = p.ik_eps;
    c.ik_lambda2_d = p.ik_lambda * p.ik_lambda;
    c.need_jp = p.mixer_w[2] != 0.0 ? 1 : 0;
    c.asin_series = (p.rot_slowdown > 0 && p.rot_slowdown <= 0.3) ? 1 : 0;
    c.order_int = (p.obst_order == std::floor(p.obst_order) && p.obst_order >= 1 && p.obst_order <= 64) ? (int)p.obst_order : 0;
}

// -------------------------------------------------------------------------------- public: lifecycle
extern "C" int vfk_version(void) { return VFK_VERSION; }

extern "C" void vfk_default_params(vfk_params* p, int n_joints) {
    if (!p) return;
    memset(p, 0, sizeof *p);
    p->ik_lambda = 0.1;
    p->ns_lambda = 0.1;
    p->dt = 0.01;
    p->speed_scale = 0.2;
    p->max_vel = 1.0;
    p->jp_kp = 1.5;
    p->jp_delta = 0.087;
    p->ns_gain = 0.5;
    p->ns_lookahead = 0.3;
    p->ns_limit_gain = 1.0;
    p->rot_slowdown = 0.09;
    p->goal_force = 1.0;
    p->obst_force = -10.0;
    p->obst_safe = 0.001;
    p->obst_order = 20.0;
    p->mixer_w[0] = p->mixer_w[1] = 1.0;
    for (int k = 0; k < 6; ++k) p->w_task[k] = 1.0;
    for (int j = 0; j < VFK_MAX_JOINTS; ++j) p->w_joint[j] = 1.0;
    p->tool[0] = p->tool[4] = p->tool[8] = 1.0;
    p->ns_mode = VFK_NS_PROJECTOR;
    p->direct_control = -1;
    p->ik_mode = VFK_IK_DLS;
    p->ik_eps = 1e-5;
    p->integrate = 1;
    (void)n_joints;
}

// Instantiated joint counts; any other chain length runs padded in the next larger one (generic pattern).
static int kernel_joints(int n) { return n <= 6 ? 6 : n <= 7 ? 7 : n <= 10 ? 10 : 17; }

static int check_params(vfk_ctx* h, const vfk_params* p) {
    if (!(p->ik_lambda >= 0) || !(p->ns_lambda >= 0)) return fail(h, VFK_ERR_INVALID, "lambda must be >= 0");
    if (p->ik_lambda == 0 && h->precision == 32 && p->ik_mode == VFK_IK_DLS)
        return fail(h, VFK_ERR_INVALID, "ik_lambda = 0 is outside the FP32 mode's domain (use precision 64)");
    if (p->ns_mode < 0 || p->ns_mode > 2) return fail(h, VFK_ERR_INVALID, "ns_mode must be 0, 1 or 2");
    if (p->ik_mode != VFK_IK_DLS && p->ik_mode != VFK_IK_TRUNCATED) return fail(h, VFK_ERR_INVALID, "ik_mode must be VFK_IK_DLS or VFK_IK_TRUNCATED");
    if (p->ik_mode == VFK_IK_TRUNCATED && h->precision != 64)
        return fail(h, VFK_ERR_UNSUPPORTED, "VFK_IK_TRUNCATED (one-sided Jacobi SVD) is built for precision 64 only");
    if (p->ik_mode == VFK_IK_TRUNCATED && !(p->ik_eps >= 0)) return fail(h, VFK_ERR_INVALID, "ik_eps must be >= 0");
    if (!(p->max_vel >= 0)) return fail(h, VFK_ERR_INVALID, "max_vel must be >= 0");
    if (p->bridge_kind < VFK_BRIDGE_LWR || p->bridge_kind > VFK_BRIDGE_ICUB)
        return fail(h, VFK_ERR_INVALID, "bridge_kind must be VFK_BRIDGE_LWR, _POWERCUBE or _ICUB");
    if (p->bridge_kind == VFK_BRIDGE_POWERCUBE && !(p->shoulder_vel[0] > 0 && p->shoulder_vel[1] < 0))
        return fail(h, VFK_ERR_INVALID, "Powercube back-end needs shoulder_vel[0] > 0 and shoulder_vel[1] < 0");
    if (!(p->obst_order > 0)) return fail(h, VFK_ERR_INVALID, "obst_order must be > 0");
    return VFK_OK;
}

extern "C" int vfk_create(vfk_handle* out, const vfk_chain_desc* chain, int precision, int device) {
    if (!out || !chain) return fail(nullptr, VFK_ERR_INVALID, "vfk_create: null argument");
    *out = nullptr;
    if (precision != 32 && precision != 64) return fail(nullptr, VFK_ERR_INVALID, "precision must be 32 or 64");
    const int n = chain->n_joints;
    if (n < 1 || n > VFK_MAX_JOINTS) return fail(nullptr, VFK_ERR_INVALID, "n_joints %d out of range", n);
    for (int j = 0; j < n; ++j) {
        if (chain->joint_type[j] < VFK_JOINT_ROTX || chain->joint_type[j] > VFK_JOINT_TRANSZ)
            return fail(nullptr, VFK_ERR_INVALID, "joint %d: type %d (fold fixed segments on the host)", j, chain->joint_type[j]);
        if (!(chain->q_lo[j] < chain->q_hi[j])) return fail(nullptr, VFK_ERR_INVALID, "joint %d: limits must satisfy lo < hi", j);
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, VFK_ERR_NO_DEVICE, "no CUDA device (%s); this library has no CPU path", cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(nullptr, VFK_ERR_INVALID, "device %d out of range (%d devices)", device, ndev);
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return fail(nullptr, VFK_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major != 10)
        return fail(nullptr, VFK_ERR_NO_DEVICE, "device %d is sm_%d%d; kernels are built for sm_100a only", device, prop.major, prop.minor);
    vfk_ctx* h = new (std::nothrow) vfk_ctx();
    if (!h) return fail(nullptr, VFK_ERR_INVALID, "out of host memory");
    h->chain = *chain;
    canonicalise_chain(h->chain, h->canon);
    h->n_kernel = kernel_joints(n);
    h->dh_chain = 1;
    for (int j = 0; j < n; ++j) {
        const double* r = h->canon.tip[j];
        const bool xtwist = r[0] == 1.0 && r[1] == 0.0 && r[2] == 0.0 && r[3] == 0.0 && r[6] == 0.0 && r[4] == r[8] && r[5] == -r[7];
        if (!xtwist || h->canon.joint_type[j] != VFK_JOINT_ROTZ) h->dh_chain = 0;
    }
    h->pattern = chain_matches<LwrPattern>(h->canon, 7) ? 1 : ((h->dh_chain && n == h->n_kernel && n >= 10) ? 2 : 0);
    h->precision = precision;
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    h->generation = 1;
    vfk_default_params(&h->params, n);
    build_const(*h, h->cf);
    build_const(*h, h->cd);
    *out = h;
    return VFK_OK;
}

extern "C" int vfk_set_params(vfk_handle h, const vfk_params* p) {
    if (!h || !p) return fail(h, VFK_ERR_INVALID, "vfk_set_params: null argument");
    int rc = check_params(h, p);
    if (rc != VFK_OK) return rc;
    h->params = *p;
    h->generation++;
    build_const(*h, h->cf);
    build_const(*h, h->cd);
    return VFK_OK;
}

extern "C" int vfk_get_params(vfk_handle h, vfk_params* out) {
    if (!h || !out) return fail(h, VFK_ERR_INVALID, "vfk_get_params: null argument");
    *out = h->params;
    return VFK_OK;
}

extern "C" int vfk_chain_pattern(vfk_handle h) { return h ? h->pattern : VFK_ERR_INVALID; }

extern "C" void vfk_destroy(vfk_handle h) { delete h; }

extern "C" const char* vfk_last_error(vfk_handle h) { return h ? h->err.c_str() : g_create_err.c_str(); }

// -------------------------------------------------------------------------------- public: step
// Device buffers: present when required, 128-byte aligned when present; the first failure in table order is reported.
struct BufferCheck {
    const void* ptr;
    const char* name;
    bool required;
};

static int check_layout(vfk_ctx* h, std::initializer_list<BufferCheck> table) {
    for (const BufferCheck& c : table) {
        if (!c.ptr) {
            if (c.required) return fail(h, VFK_ERR_INVALID, "buffer %s is required", c.name);
        } else if (reinterpret_cast<uintptr_t>(c.ptr) & 127) {
            return fail(h, VFK_ERR_INVALID, "buffer %s must be 128-byte aligned", c.name);
        }
    }
    return VFK_OK;
}

// The scene's mode and lists (vfk_step, vfk_solve, vfk_field_eval_scene).  n_obst: the per-instance count (mode 0 / 2) or
// the shared list's (mode 1).
static int check_scene(vfk_ctx* h, const vfk_buffers* b, int n_obst) {
    const int mode = b->obst_shared;
    if (mode != VFK_OBST_PER_INSTANCE && mode != VFK_OBST_SHARED && mode != VFK_OBST_MIXED)
        return fail(h, VFK_ERR_INVALID, "obst_shared must be 0, 1 or 2 (got %d)", mode);
    if (mode == VFK_OBST_SHARED && n_obst > VFK_MAX_SHARED_OBSTACLES)
        return fail(h, VFK_ERR_UNSUPPORTED, "a shared obstacle list holds at most %d obstacles (got %d)", VFK_MAX_SHARED_OBSTACLES, n_obst);
    if (mode != VFK_OBST_MIXED) return VFK_OK;
    const int ms = b->n_shared_obst;
    if (ms < 0) return fail(h, VFK_ERR_INVALID, "n_shared_obst must be >= 0 (got %d)", ms);
    if (ms > VFK_MAX_SHARED_OBSTACLES)
        return fail(h, VFK_ERR_UNSUPPORTED, "a shared obstacle list holds at most %d obstacles (got %d)", VFK_MAX_SHARED_OBSTACLES, ms);
    if (b->reserved2 != 0) return fail(h, VFK_ERR_INVALID, "vfk_buffers.reserved2 must be 0");
    // shared_obst is required even when it holds no obstacle: mode 2 without it is most likely a shared-only buffer set (a
    // dense obst) under the wrong mode, whose obst would otherwise be read as a per-instance array
    if (int rc = check_layout(h, {{b->shared_obst, "shared_obst", true}, {b->shared_obst_ext, "shared_obst_ext", false}})) return rc;
    if (n_obst > 0 && ms > 0 && (b->obst_ext == nullptr) != (b->shared_obst_ext == nullptr))
        return fail(h, VFK_ERR_INVALID, "obst_ext and shared_obst_ext go together in a mixed scene");
    return VFK_OK;
}

// The argument checks vfk_step and vfk_solve share.
static int check_step(vfk_ctx* h, const vfk_buffers* b, int64_t n, int n_obst, int k_cycles) {
    if (n < 0) return fail(h, VFK_ERR_INVALID, "n_instances must be >= 0 (got %lld)", (long long)n);
    if (n_obst < 0) return fail(h, VFK_ERR_INVALID, "n_obstacles must be >= 0");
    if (k_cycles < 1) return fail(h, VFK_ERR_INVALID, "k_cycles must be >= 1");
    if (b->n_aux < 0 || b->n_aux > 64) return fail(h, VFK_ERR_INVALID, "n_aux must be in 0..64");
    const bool need_lastvec = h->params.ns_mode == VFK_NS_CONTROL && ns_ctrl_vectors(h->chain.n_joints) > 0;
    if (int rc = check_layout(h, {{b->q, "q", true}, {b->goal, "goal", true}, {b->obst, "obst", n_obst > 0}, {b->obst_ext, "obst_ext", false},
                                  {b->aux, "aux", false}, {b->jp_ref, "jp_ref", false}, {b->jp_lo, "jp_lo", false}, {b->jp_hi, "jp_hi", false},
                                  {b->ns_in, "ns_in", false}, {b->ns_lastvec, "ns_lastvec", need_lastvec}, {b->q_cmded, "q_cmded", false},
                                  {b->qdot_vf, "qdot_vf", false}, {b->qdot_ns, "qdot_ns", false}, {b->qdot_jp, "qdot_jp", false},
                                  {b->qdot, "qdot", false}, {b->cmd, "cmd", false}, {b->pose, "pose", false}, {b->twist, "twist", false},
                                  {b->flags, "flags", false}, {b->ext_cmd[0], "ext_cmd", false}, {b->ext_cmd[1], "ext_cmd", false},
                                  {b->ext_cmd[2], "ext_cmd", false}}))
        return rc;
    if ((b->jp_lo == nullptr) != (b->jp_hi == nullptr)) return fail(h, VFK_ERR_INVALID, "jp_lo and jp_hi go together");
    return check_scene(h, b, n_obst);
}

// The scene of a call: in mode 0 (per instance) n_obst counts the instances' own lists, in mode 1 (shared) the batch-wide
// list in obst / obst_ext, in mode 2 (mixed) the own lists, with the batch-wide list in the appended fields.  Nothing below
// this point reads obst_shared.
static vfk_scene resolve_scene(const vfk_buffers* b, int n_obst) {
    const vfk_obst_list given{b->obst, b->obst_ext, n_obst};
    if (b->obst_shared == VFK_OBST_SHARED) return vfk_scene{{nullptr, nullptr, 0}, given};
    if (b->obst_shared == VFK_OBST_MIXED) return vfk_scene{given, {b->shared_obst, b->shared_obst_ext, b->n_shared_obst}};
    return vfk_scene{given, {nullptr, nullptr, 0}};
}

// The launcher (translation unit) of a call: precision, solve or step, and whether the shared list holds obstacles (the SHARED
// kernels; an empty one runs the per-instance kernels, so a mixed scene with no shared obstacle is exactly the per-instance
// call); the step kernels are split further by joint count.
static int launch_cycles(vfk_ctx* h, const CycleCall& call) {
    VFK_CUDA(h, cudaSetDevice(h->device));
    const bool f32 = h->precision == 32, shared = call.scene.shared.m > 0;
    if (call.sv && shared) return f32 ? vfk_solve_shared_f32(h, call) : vfk_solve_shared_f64(h, call);
    if (call.sv) return f32 ? vfk_solve_f32(h, call) : vfk_solve_f64(h, call);
    if (shared) return f32 ? vfk_launch_shared_f32(h, call) : vfk_launch_shared_f64(h, call);
    if (h->n_kernel <= 7) return f32 ? vfk_launch_f32_small(h, call) : vfk_launch_f64_small(h, call);
    return f32 ? vfk_launch_f32_large(h, call) : vfk_launch_f64_large(h, call);
}

static int step_impl(vfk_ctx* h, const vfk_buffers* b, int64_t n, int n_obst, int k_cycles, void* stream, const vfk_io* io) {
    if (!h || !b) return fail(h, VFK_ERR_INVALID, "vfk_step: null argument");
    int rc = check_step(h, b, n, n_obst, k_cycles);
    if (rc) return rc;
    if (n == 0) return 0;
    return launch_cycles(h, CycleCall{b, n, k_cycles, static_cast<cudaStream_t>(stream), io, nullptr, resolve_scene(b, n_obst)});
}

extern "C" int vfk_step(vfk_handle h, const vfk_buffers* b, int64_t n, int n_obst, int k_cycles, void* stream) {
    return step_impl(h, b, n, n_obst, k_cycles, stream, nullptr);
}

// -------------------------------------------------------------------------------- public: solve
extern "C" int vfk_solve(vfk_handle h, const vfk_buffers* b, int64_t n, int n_obst, int max_cycles, double tol_trans,
                         double tol_rot, int32_t* cycles_out, void* dist_out, void* stream) {
    if (!h || !b) return fail(h, VFK_ERR_INVALID, "vfk_solve: null argument");
    if (!h->params.integrate) return fail(h, VFK_ERR_INVALID, "vfk_solve needs params.integrate = 1: without the plant q never moves");
    if (max_cycles < 1) return fail(h, VFK_ERR_INVALID, "max_cycles must be >= 1");
    if (!(tol_trans >= 0) || !(tol_rot >= 0))
        return fail(h, VFK_ERR_INVALID, "tolerances must be >= 0 and not NaN (got tol_trans = %g, tol_rot = %g)", tol_trans, tol_rot);
    if (!cycles_out) return fail(h, VFK_ERR_INVALID, "vfk_solve: cycles_out is required");
    const struct { const void* p; const char* name; } per_cycle[] = {
        {b->qdot_vf, "qdot_vf"}, {b->qdot_ns, "qdot_ns"}, {b->qdot_jp, "qdot_jp"}, {b->qdot, "qdot"},
        {b->cmd, "cmd"}, {b->pose, "pose"}, {b->twist, "twist"}, {b->flags, "flags"}};
    for (const auto& o : per_cycle)
        if (o.p) return fail(h, VFK_ERR_INVALID, "vfk_solve: output %s must be NULL (a per-cycle output has no single meaning when instances stop at different cycles)", o.name);
    int rc = check_step(h, b, n, n_obst, max_cycles);
    if (rc || (rc = check_layout(h, {{cycles_out, "cycles_out", true}, {dist_out, "dist_out", false}}))) return rc;
    if (n == 0) return 0;
    const vfk_solve_io sv{tol_trans, tol_rot, cycles_out, dist_out};
    return launch_cycles(h, CycleCall{b, n, max_cycles, static_cast<cudaStream_t>(stream), nullptr, &sv, resolve_scene(b, n_obst)});
}

// The field query's launch on a resolved scene: the own lists (blocked), then the shared list (dense).
static int field_launch(vfk_ctx* h, const void* pose_in, const void* goal, const vfk_scene& sc, const void* aux, int n_aux,
                        void* twist_out, int64_t n, void* stream) {
    VFK_CUDA(h, cudaSetDevice(h->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const unsigned grid = (unsigned)((n + kSmallBlock - 1) / kSmallBlock);
    if (h->precision == 32)
        vfk_field_kernel<float><<<grid, kSmallBlock, 0, st>>>(h->cf, (const float*)pose_in, (const float*)goal,
                                                         (const Vec4<float>*)sc.own.obst, (const Vec2<float>*)sc.own.obst_ext,
                                                         (const float*)aux, n_aux, (float*)twist_out, n, sc.own.m,
                                                         (const float*)sc.shared.obst, (const float*)sc.shared.obst_ext, sc.shared.m);
    else
        vfk_field_kernel<double><<<grid, kSmallBlock, 0, st>>>(h->cd, (const double*)pose_in, (const double*)goal,
                                                          (const Vec4<double>*)sc.own.obst, (const Vec2<double>*)sc.own.obst_ext,
                                                          (const double*)aux, n_aux, (double*)twist_out, n, sc.own.m,
                                                          (const double*)sc.shared.obst, (const double*)sc.shared.obst_ext, sc.shared.m);
    VFK_CUDA(h, cudaGetLastError());
    return 1;
}

extern "C" int vfk_field_eval(vfk_handle h, const void* pose_in, const void* goal, const void* obst, const void* obst_ext,
                              const void* aux, int n_aux, void* twist_out, int64_t n, int n_obst, void* stream) {
    if (!h || !pose_in || !goal || !twist_out) return fail(h, VFK_ERR_INVALID, "vfk_field_eval: null argument");
    if (n < 0) return fail(h, VFK_ERR_INVALID, "n_instances must be >= 0");
    if (n_obst > 0 && !obst) return fail(h, VFK_ERR_INVALID, "obst is required when n_obstacles > 0");
    if (n_aux < 0 || n_aux > 64) return fail(h, VFK_ERR_INVALID, "n_aux must be in 0..64");
    if (n_aux == 0) aux = nullptr;
    if (n == 0) return 0;
    return field_launch(h, pose_in, goal, vfk_scene{{obst, obst_ext, n_obst}, {nullptr, nullptr, 0}}, aux, n_aux, twist_out, n, stream);
}

extern "C" int vfk_field_eval_scene(vfk_handle h, const void* pose_in, const vfk_buffers* b, int64_t n, int n_obst, void* twist_out,
                                    void* stream) {
    if (!h || !pose_in || !b || !b->goal || !twist_out) return fail(h, VFK_ERR_INVALID, "vfk_field_eval_scene: null argument");
    if (n < 0) return fail(h, VFK_ERR_INVALID, "n_instances must be >= 0");
    if (n_obst < 0) return fail(h, VFK_ERR_INVALID, "n_obstacles must be >= 0");
    if (b->n_aux < 0 || b->n_aux > 64) return fail(h, VFK_ERR_INVALID, "n_aux must be in 0..64");
    int rc;
    if ((rc = check_scene(h, b, n_obst)) || (rc = check_layout(h, {{b->obst, "obst", n_obst > 0}, {b->obst_ext, "obst_ext", false}})))
        return rc;
    if (n == 0) return 0;
    return field_launch(h, pose_in, b->goal, resolve_scene(b, n_obst), b->n_aux > 0 ? b->aux : nullptr, b->n_aux, twist_out, n, stream);
}

extern "C" int vfk_mix(vfk_handle h, const void* const* cmds, const double* w, int n_ports, int n_channels, void* out,
                       int32_t* nan_flags, int64_t n, void* stream) {
    if (!h || !cmds || !w || !out) return fail(h, VFK_ERR_INVALID, "vfk_mix: null argument");
    if (n_ports < 0 || n_ports > 8) return fail(h, VFK_ERR_INVALID, "n_ports must be in 0..8");
    if (n_channels < 1) return fail(h, VFK_ERR_INVALID, "n_channels must be >= 1");
    if (n < 0) return fail(h, VFK_ERR_INVALID, "n_instances must be >= 0");
    if (n == 0) return 0;
    MixArgs m;
    memset(&m, 0, sizeof m);
    m.n_ports = n_ports;
    for (int p = 0; p < n_ports; ++p) { m.cmds[p] = cmds[p]; m.w[p] = w[p]; }
    VFK_CUDA(h, cudaSetDevice(h->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int64_t tiles = (n + 31) / 32;
    int launches = 1;
    if (nan_flags) { VFK_CUDA(h, cudaMemsetAsync(nan_flags, 0, (size_t)tiles * 32 * 4, st)); }
    const unsigned grid = (unsigned)((tiles * n_channels * 32 + 255) / 256);
    if (h->precision == 32)
        vfk_mix_kernel<float><<<grid, 256, 0, st>>>(m, (float*)out, nan_flags, n_channels, tiles);
    else
        vfk_mix_kernel<double><<<grid, 256, 0, st>>>(m, (double*)out, nan_flags, n_channels, tiles);
    VFK_CUDA(h, cudaGetLastError());
    return launches;
}

extern "C" int vfk_set_vel(vfk_handle h, const void* qdot, const void* q, const void* q_cmded, double max_vel, int direct_control,
                           void* cmd_out, void* qdot_lim_out, int n_channels, int64_t n, void* stream) {
    if (!h || !qdot || !q || !cmd_out) return fail(h, VFK_ERR_INVALID, "vfk_set_vel: null argument");
    if (n_channels < 1 || n < 0 || !(max_vel >= 0)) return fail(h, VFK_ERR_INVALID, "vfk_set_vel: bad shape or max_vel");
    if (n == 0) return 0;
    VFK_CUDA(h, cudaSetDevice(h->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const unsigned grid = (unsigned)((n + 255) / 256);
    const vfk_params& p = h->params;
    const int shoulder = p.bridge_kind == VFK_BRIDGE_POWERCUBE;
    if (p.bridge_kind != VFK_BRIDGE_LWR) direct_control = 1;
    if (h->precision == 32)
        vfk_set_vel_kernel<float><<<grid, 256, 0, st>>>((const float*)qdot, (const float*)q, (const float*)q_cmded, (float*)cmd_out,
                                                       (float*)qdot_lim_out, (float)max_vel, direct_control, shoulder,
                                                       (float)p.shoulder_vel[0], (float)p.shoulder_vel[1], n_channels, n);
    else
        vfk_set_vel_kernel<double><<<grid, 256, 0, st>>>((const double*)qdot, (const double*)q, (const double*)q_cmded,
                                                        (double*)cmd_out, (double*)qdot_lim_out, max_vel, direct_control, shoulder,
                                                        p.shoulder_vel[0], p.shoulder_vel[1], n_channels, n);
    VFK_CUDA(h, cudaGetLastError());
    return 1;
}

extern "C" int vfk_monitor(vfk_handle h, const void* pose, const void* twist, const void* goal, void* state_f, int32_t* state_i,
                           void* track_out, void* dist_out, int32_t* tracking_state_out, int64_t n, void* stream) {
    if (!h || !pose || !twist || !goal || !state_f || !state_i) return fail(h, VFK_ERR_INVALID, "vfk_monitor: null argument");
    if (n < 0) return fail(h, VFK_ERR_INVALID, "n_instances must be >= 0");
    if (n == 0) return 0;
    VFK_CUDA(h, cudaSetDevice(h->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const unsigned grid = (unsigned)((n + kSmallBlock - 1) / kSmallBlock);
    if (h->precision == 32)
        vfk_monitor_kernel<float><<<grid, kSmallBlock, 0, st>>>((const float*)pose, (const float*)twist, (const float*)goal,
                                                               (float*)state_f, state_i, (float*)track_out, (float*)dist_out,
                                                               tracking_state_out, n);
    else
        vfk_monitor_kernel<double><<<grid, kSmallBlock, 0, st>>>((const double*)pose, (const double*)twist, (const double*)goal,
                                                                (double*)state_f, state_i, (double*)track_out, (double*)dist_out,
                                                                tracking_state_out, n);
    VFK_CUDA(h, cudaGetLastError());
    return 1;
}

// -------------------------------------------------------------------------------- public: layout conversion
template <typename V>
static cudaError_t run_pack(const void* dense, int64_t dense_ld, void* blocked, int C, int64_t n, bool unpack, cudaStream_t st) {
    const int64_t tiles = (n + 31) / 32;
    const unsigned grid = (unsigned)((tiles * C * 32 + 255) / 256);
    if (unpack)
        vfk_unpack_kernel<V><<<grid, 256, 0, st>>>((const V*)blocked, (V*)const_cast<void*>(dense), dense_ld, C, n, tiles);
    else
        vfk_pack_kernel<V><<<grid, 256, 0, st>>>((const V*)dense, dense_ld, (V*)blocked, C, n, tiles);
    return cudaGetLastError();
}

// obstacles (width 4): dense [M][ld] {x, y, z, radius} <-> the pair-interleaved blocked array (vfk.h, ObstPairs)
template <typename T>
static cudaError_t run_pack_obst(const void* dense, int64_t dense_ld, void* blocked, int M, int64_t n, bool unpack, cudaStream_t st) {
    const int64_t tiles = (n + 31) / 32;
    const unsigned grid = (unsigned)((tiles * ((M + 1) / 2) * 32 + 255) / 256);
    if (unpack)
        vfk_unpack_obst_kernel<T><<<grid, 256, 0, st>>>((const Vec4<T>*)blocked, (Vec4<T>*)const_cast<void*>(dense), dense_ld, M, n, tiles);
    else
        vfk_pack_obst_kernel<T><<<grid, 256, 0, st>>>((const Vec4<T>*)dense, dense_ld, (Vec4<T>*)blocked, M, n, tiles);
    return cudaGetLastError();
}

// width = scalars per element: 1 (per-instance components), 2 (obstacle ext) or 4 (obstacles);
// dense_ld = row pitch of the dense array in elements (>= n; lets a column range of a larger array be converted)
static int pack_dispatch(vfk_ctx* h, const void* dense, void* blocked, int C, int width, int64_t n, bool unpack,
                         cudaStream_t st, int64_t dense_ld = -1) {
    if (!dense || !blocked) return fail(h, VFK_ERR_INVALID, "vfk_pack/unpack: null buffer");
    if (C < 1 || n < 0) return fail(h, VFK_ERR_INVALID, "vfk_pack/unpack: bad shape");
    if (n == 0) return 0;
    if (dense_ld < 0) dense_ld = n;
    cudaError_t e;
    const bool f = h->precision == 32;
    if (width == 1) e = f ? run_pack<float>(dense, dense_ld, blocked, C, n, unpack, st) : run_pack<double>(dense, dense_ld, blocked, C, n, unpack, st);
    else if (width == 2) e = f ? run_pack<Vec2<float>>(dense, dense_ld, blocked, C, n, unpack, st) : run_pack<Vec2<double>>(dense, dense_ld, blocked, C, n, unpack, st);
    else if (width == 4) e = f ? run_pack_obst<float>(dense, dense_ld, blocked, C, n, unpack, st) : run_pack_obst<double>(dense, dense_ld, blocked, C, n, unpack, st);
    else return fail(h, VFK_ERR_INVALID, "vfk_pack/unpack: width must be 1, 2 or 4");
    if (e != cudaSuccess) return fail(h, VFK_ERR_CUDA, "layout kernel: %s", cudaGetErrorString(e));
    return 1;
}

extern "C" int vfk_pack(vfk_handle h, const void* dense, void* blocked, int comps, int width, int64_t n, void* stream) {
    if (!h) return fail(h, VFK_ERR_INVALID, "vfk_pack: null handle");
    VFK_CUDA(h, cudaSetDevice(h->device));
    return pack_dispatch(h, dense, blocked, comps, width, n, false, static_cast<cudaStream_t>(stream));
}

extern "C" int vfk_unpack(vfk_handle h, const void* blocked, void* dense, int comps, int width, int64_t n, void* stream) {
    if (!h) return fail(h, VFK_ERR_INVALID, "vfk_unpack: null handle");
    VFK_CUDA(h, cudaSetDevice(h->device));
    return pack_dispatch(h, dense, const_cast<void*>(blocked), comps, width, n, true, static_cast<cudaStream_t>(stream));
}

// -------------------------------------------------------------------------------- public: host-buffer sessions
// Host arrays are dense SoA ([comps][n]; obstacles [M][n][4]); the session keeps a dense device staging
// area and converts to / from the kernels' tile-blocked layout on the GPU (vfk_pack / vfk_unpack kernels).
constexpr int kMaxSessionChunks = 32;

struct vfk_session_s {
    vfk_ctx* h;
    int device;                      // copied from the handle: destroy must not touch a handle that may be gone
    int64_t n, tiles;
    int n_obst, has_ext, N, n_aux;
    size_t es;                       // element size
    cudaStream_t stream;
    cudaStream_t pipe[3];            // chunk pipeline of vfk_session_cycle: [0] H2D, [1] kernels, [2] D2H
    cudaEvent_t ev_up[kMaxSessionChunks], ev_done[kMaxSessionChunks], ev_fork, ev_join[2];
    char* dev;                       // one device slab
    size_t dev_bytes;
    vfk_buffers b;                   // blocked device buffers
    void* stage_in;                  // dense staging, big enough for the largest upload
    void* stage_out;                 // dense staging for outputs (max(N, 12) rows)
    bool have_jp_ref, have_ns_in, have_jp_lim;
    bool en_vf, en_ns, en_jp, en_cmd, en_pose, en_twist;   // optional per-controller outputs (off by default)
    void *d_jp_ref, *d_ns_in, *d_jp_lo, *d_jp_hi;
    void *d_cycles, *d_dist;         // vfk_session_solve's results: cycles [1] int32, dist [2]
    char* aux_dev;                   // auxiliary field records (blocked + dense staging), grown on demand
    char* shared_dev;                // shared scene: dense [VFK_MAX_SHARED_OBSTACLES][4], then [..][2] ext; allocated on first use
    int shared_m;                    // obstacles in it
    bool shared_ext;                 // it has ext rows
    int obst_mode;                   // VFK_OBST_*: the lists cycles and solves use
    char* pin;                       // pinned host staging: q in (N rows), qdot / q out (2N rows), flags
    size_t pin_bytes;
    int launches;                    // kernels launched by the last call
    uint64_t generation;             // bumped by every setter that changes what a cycle does
    // cached CUDA graph of one vfk_session_cycle (the pipeline is ~30-100 API calls; one graph launch replaces them)
    cudaGraphExec_t graph_exec;
    int graph_launches;
    struct { const void *src_q, *dst_qd, *dst_qo, *dst_fl; int k; uint64_t hgen, sgen; } graph_key;
};

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static void session_release(vfk_session_s* s);

// Smallest batch for which vfk_session_cycle reads / writes page-locked caller buffers directly from the kernel.
constexpr int64_t kDirectMinInstances = 1024;

extern "C" int vfk_session_create(vfk_handle h, int64_t n, int n_obst, int with_obst_ext, vfk_session* out) {
    if (!h || !out) return fail(h, VFK_ERR_INVALID, "vfk_session_create: null argument");
    *out = nullptr;
    if (n < 1) return fail(h, VFK_ERR_INVALID, "n_instances must be >= 1");
    if (n_obst < 0) return fail(h, VFK_ERR_INVALID, "n_obstacles must be >= 0");
    VFK_CUDA(h, cudaSetDevice(h->device));
    vfk_session_s* s = new (std::nothrow) vfk_session_s();
    if (!s) return fail(h, VFK_ERR_INVALID, "out of host memory");
    memset(&s->b, 0, sizeof s->b);
    s->h = h;
    s->device = h->device;
    s->n = n;
    s->tiles = (n + 31) / 32;
    s->n_obst = n_obst;
    s->has_ext = with_obst_ext ? 1 : 0;
    s->N = h->chain.n_joints;
    s->es = h->precision == 32 ? 4 : 8;
    const int N = s->N;
    const size_t row = align_up((size_t)s->tiles * 32 * s->es, 128);     // one component over all tiles
    const size_t obst_rows = (size_t)((n_obst + 1) & ~1) * 4 + (size_t)n_obst * (s->has_ext ? 2 : 0);
    // blocked: q N, goal 13, obst, jp_ref N, ns_in N, lastvec N, qdot_vf N, qdot_ns N, qdot_jp N, qdot N, cmd N, pose 12, twist 6, flags 1,
    // solve cycles 1 + dist 2
    const int lv_rows = (ns_ctrl_vectors(N) > 0 ? ns_ctrl_vectors(N) : 1) * N;   // sign-continuity state: [min(4, N - 6)][N]
    const size_t rows = (size_t)N * 10 + lv_rows + 13 + obst_rows + 12 + 6 + 1 + 3;
    const size_t stage_in_rows = obst_rows > (size_t)(N > 13 ? N : 13) ? obst_rows : (size_t)(N > 13 ? N : 13);
    const size_t first_out = (size_t)(lv_rows > 12 ? lv_rows : 12);
    const size_t stage_out_rows = first_out + (size_t)N;                          // qdot (or a read()) + q_out
    s->dev_bytes = (rows + stage_in_rows + stage_out_rows) * row;
    cudaError_t e = cudaMalloc((void**)&s->dev, s->dev_bytes);
    if (e != cudaSuccess) { s->dev = nullptr; session_release(s); return fail(h, VFK_ERR_CUDA, "cudaMalloc(%zu): %s", s->dev_bytes, cudaGetErrorString(e)); }
    e = cudaMemset(s->dev, 0, s->dev_bytes);
    char* p = s->dev;
    auto take = [&](size_t nrows) { char* r = p; p += nrows * row; return (void*)r; };
    s->b.q = take(N);
    s->b.goal = take(13);
    s->b.obst = n_obst ? take((size_t)((n_obst + 1) & ~1) * 4) : nullptr;     // whole pairs
    s->b.obst_ext = (n_obst && s->has_ext) ? take((size_t)n_obst * 2) : nullptr;
    s->d_jp_ref = take(N);
    s->d_jp_lo = take(N);
    s->d_jp_hi = take(N);
    s->d_ns_in = take(N);
    s->b.ns_lastvec = take(lv_rows);
    s->b.qdot_vf = take(N);
    s->b.qdot_ns = take(N);
    s->b.qdot_jp = take(N);
    s->b.qdot = take(N);
    s->b.cmd = take(N);
    s->b.pose = take(12);
    s->b.twist = take(6);
    s->b.flags = (int32_t*)take(1);
    s->d_cycles = take(1);
    s->d_dist = take(2);
    s->stage_in = take(stage_in_rows);
    s->stage_out = take(stage_out_rows);
    s->have_jp_ref = s->have_ns_in = s->have_jp_lim = false;
    s->en_vf = s->en_ns = s->en_jp = s->en_cmd = s->en_pose = s->en_twist = false;
    s->launches = 0;
    s->n_aux = 0;
    s->aux_dev = nullptr;
    s->shared_dev = nullptr;
    s->shared_m = 0;
    s->shared_ext = false;
    s->obst_mode = VFK_OBST_PER_INSTANCE;
    s->generation = 1;
    s->graph_exec = nullptr;
    s->graph_launches = 0;
    memset(&s->graph_key, 0, sizeof s->graph_key);
    s->pin_bytes = (size_t)N * 3 * (size_t)n * s->es + (size_t)n * 4;
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
    for (int k = 0; k < 3 && e == cudaSuccess; ++k) e = cudaStreamCreateWithFlags(&s->pipe[k], cudaStreamNonBlocking);
    for (int k = 0; k < kMaxSessionChunks && e == cudaSuccess; ++k) {
        e = cudaEventCreateWithFlags(&s->ev_up[k], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_done[k], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_fork, cudaEventDisableTiming);
    for (int k = 0; k < 2 && e == cudaSuccess; ++k) e = cudaEventCreateWithFlags(&s->ev_join[k], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMallocHost((void**)&s->pin, s->pin_bytes);
    if (e != cudaSuccess) {
        session_release(s);
        return fail(h, VFK_ERR_CUDA, "session allocation: %s", cudaGetErrorString(e));
    }
    *out = s;
    return VFK_OK;
}

// dense host [rows][n] (x width scalars) -> blocked device array
static int upload_blocked(vfk_session_s* s, void* dst_blocked, const void* src_host, int comps, int width) {
    vfk_ctx* h = s->h;
    VFK_CUDA(h, cudaSetDevice(h->device));
    const size_t bytes = (size_t)comps * width * (size_t)s->n * s->es;
    VFK_CUDA(h, cudaMemcpyAsync(s->stage_in, src_host, bytes, cudaMemcpyHostToDevice, s->stream));
    int rc = pack_dispatch(h, s->stage_in, dst_blocked, comps, width, s->n, false, s->stream);
    if (rc < 0) return rc;
    s->launches += rc;
    VFK_CUDA(h, cudaStreamSynchronize(s->stream));
    return VFK_OK;
}

extern "C" int vfk_session_set_goal(vfk_session s, const void* g) {
    if (!s || !g) return fail(s ? s->h : nullptr, VFK_ERR_INVALID, "vfk_session_set_goal: null argument");
    return upload_blocked(s, const_cast<void*>(s->b.goal), g, 13, 1);
}

// host obstacles: dense [M][n][4] (x, y, z, radius per instance); ext: dense [M][n][2] (safe, order)
extern "C" int vfk_session_set_obstacles(vfk_session s, const void* o, const void* ext) {
    if (!s) return fail(nullptr, VFK_ERR_INVALID, "vfk_session_set_obstacles: null session");
    if (s->n_obst == 0) return VFK_OK;
    if (!o) return fail(s->h, VFK_ERR_INVALID, "vfk_session_set_obstacles: null argument");
    if (s->has_ext && !ext) return fail(s->h, VFK_ERR_INVALID, "vfk_session_set_obstacles: session was created with obstacle ext rows");
    if (s->obst_mode != VFK_OBST_PER_INSTANCE) { s->obst_mode = VFK_OBST_PER_INSTANCE; s->generation++; }  // back to the per-instance scene
    int rc = upload_blocked(s, const_cast<void*>(s->b.obst), o, s->n_obst, 4);
    if (rc == VFK_OK && s->has_ext) rc = upload_blocked(s, const_cast<void*>(s->b.obst_ext), ext, s->n_obst, 2);
    return rc;
}

// one scene for every instance: dense [M][4] host list (ext [M][2] or NULL) -> the session's shared-scene buffer
extern "C" int vfk_session_set_shared_obstacles(vfk_session s, const void* o, const void* ext, int M) {
    if (!s) return fail(nullptr, VFK_ERR_INVALID, "vfk_session_set_shared_obstacles: null session");
    vfk_ctx* h = s->h;
    if (M < 0) return fail(h, VFK_ERR_INVALID, "n_obstacles must be >= 0");
    if (M > VFK_MAX_SHARED_OBSTACLES)
        return fail(h, VFK_ERR_UNSUPPORTED, "a shared obstacle list holds at most %d obstacles (got %d)", VFK_MAX_SHARED_OBSTACLES, M);
    if (M > 0 && !o) return fail(h, VFK_ERR_INVALID, "vfk_session_set_shared_obstacles: null obstacle list");
    VFK_CUDA(h, cudaSetDevice(h->device));
    const size_t list = (size_t)VFK_MAX_SHARED_OBSTACLES * 4 * s->es;
    if (!s->shared_dev) VFK_CUDA(h, cudaMalloc((void**)&s->shared_dev, list + (size_t)VFK_MAX_SHARED_OBSTACLES * 2 * s->es));
    if (M > 0) {
        VFK_CUDA(h, cudaMemcpyAsync(s->shared_dev, o, (size_t)M * 4 * s->es, cudaMemcpyHostToDevice, s->stream));
        if (ext) VFK_CUDA(h, cudaMemcpyAsync(s->shared_dev + list, ext, (size_t)M * 2 * s->es, cudaMemcpyHostToDevice, s->stream));
        VFK_CUDA(h, cudaStreamSynchronize(s->stream));
    }
    s->obst_mode = VFK_OBST_SHARED;
    s->shared_m = M;
    s->shared_ext = ext != nullptr;
    s->generation++;
    return VFK_OK;
}

// Which lists the session's calls use (vfk_session_use_obstacles): the per-instance arrays, the shared list or both.
extern "C" int vfk_session_use_obstacles(vfk_session s, int mode) {
    if (!s) return fail(nullptr, VFK_ERR_INVALID, "vfk_session_use_obstacles: null session");
    vfk_ctx* h = s->h;
    if (mode != VFK_OBST_PER_INSTANCE && mode != VFK_OBST_SHARED && mode != VFK_OBST_MIXED)
        return fail(h, VFK_ERR_INVALID, "vfk_session_use_obstacles: mode must be 0, 1 or 2 (got %d)", mode);
    if (mode != VFK_OBST_PER_INSTANCE && !s->shared_dev)
        return fail(h, VFK_ERR_INVALID, "vfk_session_use_obstacles: no shared obstacle list was set (vfk_session_set_shared_obstacles)");
    if (mode == VFK_OBST_MIXED && s->n_obst == 0)
        return fail(h, VFK_ERR_INVALID, "vfk_session_use_obstacles: a mixed scene needs a session created with n_obstacles > 0");
    if (mode == VFK_OBST_MIXED && s->shared_m > 0 && (s->has_ext != 0) != s->shared_ext)
        return fail(h, VFK_ERR_INVALID, "vfk_session_use_obstacles: the per-instance and shared lists' ext rows go together");
    s->obst_mode = mode;
    s->generation++;
    return VFK_OK;
}

// What a session call's view holds besides q, goal, the scene and the inputs that are set: every output
// (vfk_session_buffers), qdot and the enabled outputs (a cycle), or none (a solve).
enum class SessionOutputs { all, enabled, none };

// The blocked device view of a session call in `v`: the scene of the session's mode (the shared list whole, never offset by a
// tile range), the per-instance inputs that are set and the outputs `outs` selects, a cycle's flags only when `want_flags`.
// Returns the call's n_obstacles argument: the shared count in mode 1, the per-instance one otherwise.
static int session_view(const vfk_session_s* s, SessionOutputs outs, bool want_flags, vfk_buffers* v) {
    *v = s->b;
    v->jp_ref = s->have_jp_ref ? s->d_jp_ref : nullptr;
    v->jp_lo = s->have_jp_lim ? s->d_jp_lo : nullptr;
    v->jp_hi = s->have_jp_lim ? s->d_jp_hi : nullptr;
    v->ns_in = s->have_ns_in ? s->d_ns_in : nullptr;
    const bool all = outs == SessionOutputs::all, none = outs == SessionOutputs::none;
    auto keep = [&](bool enabled) { return all || (enabled && !none); };
    if (!keep(true)) v->qdot = nullptr;
    if (!keep(s->en_vf)) v->qdot_vf = nullptr;
    if (!keep(s->en_ns)) v->qdot_ns = nullptr;
    if (!keep(s->en_jp)) v->qdot_jp = nullptr;
    if (!keep(s->en_cmd)) v->cmd = nullptr;
    if (!keep(s->en_pose)) v->pose = nullptr;
    if (!keep(s->en_twist)) v->twist = nullptr;
    if (!keep(want_flags)) v->flags = nullptr;
    if (s->obst_mode == VFK_OBST_PER_INSTANCE) return s->n_obst;
    const void* ext = s->shared_ext ? s->shared_dev + (size_t)VFK_MAX_SHARED_OBSTACLES * 4 * s->es : nullptr;
    v->obst_shared = s->obst_mode;
    if (s->obst_mode == VFK_OBST_SHARED) {
        v->obst = s->shared_dev;
        v->obst_ext = ext;
        return s->shared_m;
    }
    v->shared_obst = s->shared_dev;
    v->shared_obst_ext = ext;
    v->n_shared_obst = s->shared_m;
    return s->n_obst;
}

extern "C" int vfk_session_set_aux(vfk_session s, const void* aux, int n_aux) {
    if (!s) return fail(nullptr, VFK_ERR_INVALID, "vfk_session_set_aux: null session");
    vfk_ctx* h = s->h;
    if (n_aux < 0 || n_aux > 64) return fail(h, VFK_ERR_INVALID, "n_aux must be in 0..64");
    VFK_CUDA(h, cudaSetDevice(h->device));
    s->generation++;
    if (!aux || n_aux == 0) { s->b.n_aux = 0; return VFK_OK; }
    const size_t row = align_up((size_t)s->tiles * 32 * s->es, 128);
    if (n_aux > s->n_aux) {                                   // grow the dedicated buffers (blocked + dense staging)
        s->b.aux = nullptr;                                   // nothing may point at the old block once it is gone
        s->b.n_aux = 0;
        s->n_aux = 0;
        char* old = s->aux_dev;
        s->aux_dev = nullptr;
        if (old) VFK_CUDA(h, cudaFree(old));
        VFK_CUDA(h, cudaMalloc((void**)&s->aux_dev, 2 * (size_t)n_aux * 12 * row));
        s->n_aux = n_aux;
    }
    char* blocked = s->aux_dev;
    char* dense = s->aux_dev + (size_t)s->n_aux * 12 * row;
    VFK_CUDA(h, cudaMemcpyAsync(dense, aux, (size_t)n_aux * 12 * s->n * s->es, cudaMemcpyHostToDevice, s->stream));
    int rc = pack_dispatch(h, dense, blocked, n_aux * 12, 1, s->n, false, s->stream);
    if (rc < 0) return rc;
    VFK_CUDA(h, cudaStreamSynchronize(s->stream));
    s->b.aux = blocked;
    s->b.n_aux = n_aux;
    return VFK_OK;
}

extern "C" int vfk_session_set_q(vfk_session s, const void* q) {
    if (!s || !q) return fail(s ? s->h : nullptr, VFK_ERR_INVALID, "vfk_session_set_q: null argument");
    return upload_blocked(s, s->b.q, q, s->N, 1);
}

extern "C" int vfk_session_set_jp_ref(vfk_session s, const void* r) {
    if (!s) return fail(nullptr, VFK_ERR_INVALID, "vfk_session_set_jp_ref: null session");
    s->have_jp_ref = r != nullptr;
    s->generation++;
    if (!r) return VFK_OK;
    return upload_blocked(s, s->d_jp_ref, r, s->N, 1);
}

extern "C" int vfk_session_set_jp_limits(vfk_session s, const void* lo, const void* hi) {
    if (!s) return fail(nullptr, VFK_ERR_INVALID, "vfk_session_set_jp_limits: null session");
    if ((lo == nullptr) != (hi == nullptr)) return fail(s->h, VFK_ERR_INVALID, "vfk_session_set_jp_limits: lo and hi go together");
    s->have_jp_lim = lo != nullptr;
    s->generation++;
    if (!lo) return VFK_OK;
    int rc = upload_blocked(s, s->d_jp_lo, lo, s->N, 1);
    if (rc == VFK_OK) rc = upload_blocked(s, s->d_jp_hi, hi, s->N, 1);
    return rc;
}

extern "C" int vfk_session_set_ns_input(vfk_session s, const void* x) {
    if (!s) return fail(nullptr, VFK_ERR_INVALID, "vfk_session_set_ns_input: null session");
    s->have_ns_in = x != nullptr;
    s->generation++;
    if (!x) return VFK_OK;
    return upload_blocked(s, s->d_ns_in, x, s->h->params.ns_mode == VFK_NS_CONTROL ? 4 : s->N, 1);
}

// Offset every per-instance buffer of a blocked view to the tile range starting at tile0 (a shared list stays whole; a mixed
// scene's own list is offset like any per-instance buffer).  ns_comps: components of ns_in (4 or N).
static vfk_buffers offset_view(const vfk_buffers& b, int64_t tile0, int N, int M, int ns_comps, size_t es) {
    vfk_buffers o = b;
    auto off = [&](const void* p, size_t comps) -> void* {
        return p ? (void*)((char*)const_cast<void*>(p) + (size_t)tile0 * comps * 32 * es) : nullptr;
    };
    o.q = off(b.q, N); o.goal = off(b.goal, 13);
    if (b.obst_shared != VFK_OBST_SHARED) { o.obst = off(b.obst, (size_t)((M + 1) & ~1) * 4); o.obst_ext = off(b.obst_ext, (size_t)M * 2); }
    o.aux = off(b.aux, (size_t)b.n_aux * 12);
    o.jp_ref = off(b.jp_ref, N); o.jp_lo = off(b.jp_lo, N); o.jp_hi = off(b.jp_hi, N); o.ns_in = off(b.ns_in, ns_comps); o.ns_lastvec = off(b.ns_lastvec, (size_t)(ns_ctrl_vectors(N) > 0 ? ns_ctrl_vectors(N) : 1) * N); o.q_cmded = off(b.q_cmded, N);
    for (int e = 0; e < 3; ++e) o.ext_cmd[e] = off(b.ext_cmd[e], N);
    o.qdot_vf = off(b.qdot_vf, N); o.qdot_ns = off(b.qdot_ns, N); o.qdot_jp = off(b.qdot_jp, N); o.qdot = off(b.qdot, N);
    o.cmd = off(b.cmd, N); o.pose = off(b.pose, 12); o.twist = off(b.twist, 6);
    o.flags = b.flags ? b.flags + tile0 * 32 : nullptr;
    return o;
}

// Enqueue one cycle's pipeline (uploads, layout kernels, cycle kernels, downloads) on the session's streams.
// Used eagerly and under stream capture; returns the number of kernels enqueued.
static int enqueue_cycle(vfk_session_s* s, const char* src_q, int k_cycles, char* dst_qd, char* dst_qo, char* dst_fl,
                         bool want_flags, int n_chunks) {
    vfk_ctx* h = s->h;
    const int N = s->N;
    const size_t es = s->es;
    vfk_buffers b;
    const int M = session_view(s, SessionOutputs::enabled, want_flags, &b);
    const int ns_comps = h->params.ns_mode == VFK_NS_CONTROL ? 4 : N;
    const bool piped = n_chunks > 1;
    cudaStream_t st_up = piped ? s->pipe[0] : s->pipe[1], st_k = s->pipe[1], st_dn = piped ? s->pipe[2] : s->pipe[1];
    const int64_t tiles_per_chunk = (s->tiles + n_chunks - 1) / n_chunks;
    char* stage_q = (char*)s->stage_in;                         // dense [N][n]
    char* stage_qd = (char*)s->stage_out;                       // dense [N][n]
    const size_t lv_rows = (size_t)(ns_ctrl_vectors(N) > 0 ? ns_ctrl_vectors(N) : 1) * N;
    char* stage_qo = (char*)s->stage_out + (lv_rows > 12 ? lv_rows : 12) * (align_up((size_t)s->tiles * 32 * es, 128));
    const size_t pitch = (size_t)s->n * es;
    int launches = 0, rc;
    for (int c = 0; c < n_chunks; ++c) {
        const int64_t t0 = (int64_t)c * tiles_per_chunk;
        if (t0 >= s->tiles) break;
        const int64_t t1 = t0 + tiles_per_chunk < s->tiles ? t0 + tiles_per_chunk : s->tiles;
        const int64_t i0 = t0 * 32;
        const int64_t cnt = (t1 * 32 < s->n ? t1 * 32 : s->n) - i0;
        vfk_buffers v = offset_view(b, t0, N, M, ns_comps, es);
        if (src_q) {
            VFK_CUDA(h, cudaMemcpy2DAsync(stage_q + i0 * es, pitch, src_q + i0 * es, pitch, (size_t)cnt * es, N,
                                          cudaMemcpyHostToDevice, st_up));
            if (piped) {
                VFK_CUDA(h, cudaEventRecord(s->ev_up[c], st_up));
                VFK_CUDA(h, cudaStreamWaitEvent(st_k, s->ev_up[c], 0));
            }
            if ((rc = pack_dispatch(h, stage_q + i0 * es, v.q, N, 1, cnt, false, st_k, s->n)) < 0) return rc;
            launches += rc;
        }
        if ((rc = vfk_step(h, &v, cnt, M, k_cycles, st_k)) < 0) return rc;
        launches += rc;
        if (dst_qd) {
            if ((rc = pack_dispatch(h, stage_qd + i0 * es, v.qdot, N, 1, cnt, true, st_k, s->n)) < 0) return rc;
            launches += rc;
        }
        if (dst_qo) {
            if ((rc = pack_dispatch(h, stage_qo + i0 * es, v.q, N, 1, cnt, true, st_k, s->n)) < 0) return rc;
            launches += rc;
        }
        if (piped) {
            VFK_CUDA(h, cudaEventRecord(s->ev_done[c], st_k));
            VFK_CUDA(h, cudaStreamWaitEvent(st_dn, s->ev_done[c], 0));
        }
        if (dst_qd)
            VFK_CUDA(h, cudaMemcpy2DAsync(dst_qd + i0 * es, pitch, stage_qd + i0 * es, pitch, (size_t)cnt * es, N,
                                          cudaMemcpyDeviceToHost, st_dn));
        if (dst_qo)
            VFK_CUDA(h, cudaMemcpy2DAsync(dst_qo + i0 * es, pitch, stage_qo + i0 * es, pitch, (size_t)cnt * es, N,
                                          cudaMemcpyDeviceToHost, st_dn));
        if (dst_fl)         // one component: blocked == dense
            VFK_CUDA(h, cudaMemcpyAsync(dst_fl + i0 * 4, s->b.flags + i0, (size_t)cnt * 4, cudaMemcpyDeviceToHost, st_dn));
    }
    return launches;
}

// Is p page-locked host memory (cudaHostAlloc / cudaHostRegister / torch pinned memory)?  `mapped` gets its device address,
// or null.
static bool host_pinned(const void* p, void** mapped = nullptr) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    if (mapped) *mapped = at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
    return at.type == cudaMemoryTypeHost;
}

// Direct host I/O (zero-copy): when the caller's q_in / qdot_out are page-locked and the batch is tile-aligned, ONE
// kernel launch reads the q tiles straight from host memory through TMA (N x 128 B bulk copies per tile, prefetched one
// tile ahead like every other stream of the kernel) and stores qdot straight back with coalesced 128 B writes: no
// staging copies, no layout kernels, and the PCIe reads, the arithmetic and the PCIe writes overlap at tile
// granularity instead of chunk granularity.  Measured on B200, 1 M instances (scripts/e2e_direct.sh): 0.79 ms per call
// against 0.91 ms for the chunked copy pipeline below; hybrids (kernel reads + DMA writes 1.04 ms, DMA reads + kernel
// writes 0.83 ms) lose to both-direct.  SM-issued PCIe traffic runs at 51 / 52 GB/s one way whatever the request size
// and ~37 GB/s each way when both directions are busy (scripts/pcie_probe.cu), which is where this path sits.
// VFK_SESSION_DIRECT=0 selects the copy pipeline.
static int session_cycle_direct(vfk_session_s* s, void* dq, void* dqd, int k_cycles, char* dst_qo, char* dst_fl, bool want_flags) {
    vfk_ctx* h = s->h;
    vfk_buffers b;
    const int M = session_view(s, SessionOutputs::enabled, want_flags, &b);
    cudaStream_t st = s->pipe[1];
    vfk_io io;
    io.q_src = dq; io.q_src_ld = s->n;
    io.qdot = dqd; io.qdot_ld = dqd ? s->n : 0;
    int rc = step_impl(h, &b, s->n, M, k_cycles, st, &io);
    if (rc < 0) return rc;
    int launches = rc;
    if (dst_qo) {
        char* stage_qo = (char*)s->stage_out;
        if ((rc = pack_dispatch(h, stage_qo, b.q, s->N, 1, s->n, true, st, s->n)) < 0) return rc;
        launches += rc;
        VFK_CUDA(h, cudaMemcpyAsync(dst_qo, stage_qo, (size_t)s->N * (size_t)s->n * s->es, cudaMemcpyDeviceToHost, st));
    }
    if (dst_fl) VFK_CUDA(h, cudaMemcpyAsync(dst_fl, s->b.flags, (size_t)s->n * 4, cudaMemcpyDeviceToHost, st));
    VFK_CUDA(h, cudaStreamSynchronize(st));
    s->launches = launches;
    return launches;
}

static int session_cycle_pipeline(vfk_session_s* s, const char* src_q, int k_cycles, char* dst_qd, char* dst_qo, char* dst_fl,
                                  bool want_flags) {
    vfk_ctx* h = s->h;
    // Chunk pipeline: a three-stage software pipeline over tile-aligned chunks.  All uploads go back to back on the
    // H2D stream, the kernels of chunk c wait for its upload on the compute stream, and its downloads wait for the
    // kernels on the D2H stream, so the two DMA engines (PCIe is full duplex) and the SMs all stay busy.
    // (measured on B200, 1 M instances: 1 chunk 1.26 ms, 4 chunks 0.90 ms, 8 chunks 0.96 ms, 16 chunks 1.05 ms per call;
    //  the floor set by the two concurrent 29 MB PCIe transfers is 0.62 ms)
    int n_chunks = (int)(s->n / 65536);
    if (n_chunks > 4) n_chunks = 4;
    if (n_chunks < 1) n_chunks = 1;
    if ((int64_t)n_chunks > s->tiles) n_chunks = (int)s->tiles;

    // The pipeline is dozens of API calls; repeated calls with the same buffers replay ONE captured CUDA graph.
    // The first call with a given (buffers, K, parameter generation) runs eagerly (it also warms the launch-plan
    // caches), the second captures, later ones only launch the graph.
    const bool use_graph = n_chunks > 1;
    auto& key = s->graph_key;
    const bool same = key.src_q == src_q && key.dst_qd == dst_qd && key.dst_qo == dst_qo && key.dst_fl == dst_fl &&
                      key.k == k_cycles && key.hgen == h->generation && key.sgen == s->generation;
    int launches = 0;
    cudaStream_t origin = s->pipe[1];
    if (use_graph && same && s->graph_exec) {
        VFK_CUDA(h, cudaGraphLaunch(s->graph_exec, origin));
        launches = s->graph_launches;
    } else if (use_graph && same) {
        cudaGraph_t graph = nullptr;
        VFK_CUDA(h, cudaStreamBeginCapture(origin, cudaStreamCaptureModeThreadLocal));
        cudaError_t ce = cudaEventRecord(s->ev_fork, origin);                       // fork the two DMA streams
        if (ce == cudaSuccess) ce = cudaStreamWaitEvent(s->pipe[0], s->ev_fork, 0);
        if (ce == cudaSuccess) ce = cudaStreamWaitEvent(s->pipe[2], s->ev_fork, 0);
        int rc = ce == cudaSuccess ? enqueue_cycle(s, src_q, k_cycles, dst_qd, dst_qo, dst_fl, want_flags, n_chunks) : -1;
        if (ce == cudaSuccess) ce = cudaEventRecord(s->ev_join[0], s->pipe[0]);     // join them back
        if (ce == cudaSuccess) ce = cudaEventRecord(s->ev_join[1], s->pipe[2]);
        if (ce == cudaSuccess) ce = cudaStreamWaitEvent(origin, s->ev_join[0], 0);
        if (ce == cudaSuccess) ce = cudaStreamWaitEvent(origin, s->ev_join[1], 0);
        cudaError_t ee = cudaStreamEndCapture(origin, &graph);
        if (rc < 0 || ce != cudaSuccess || ee != cudaSuccess || !graph) {
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            if (rc < 0 && ce == cudaSuccess) return rc;
            return fail(h, VFK_ERR_CUDA, "graph capture of the session pipeline failed: %s",
                        cudaGetErrorString(ce != cudaSuccess ? ce : ee));
        }
        if (s->graph_exec) { cudaGraphExecDestroy(s->graph_exec); s->graph_exec = nullptr; }
        cudaError_t ie = cudaGraphInstantiate(&s->graph_exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) { s->graph_exec = nullptr; return fail(h, VFK_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(ie)); }
        s->graph_launches = rc;
        VFK_CUDA(h, cudaGraphLaunch(s->graph_exec, origin));
        launches = rc;
    } else {
        if (s->graph_exec) { cudaGraphExecDestroy(s->graph_exec); s->graph_exec = nullptr; }
        key.src_q = src_q; key.dst_qd = dst_qd; key.dst_qo = dst_qo; key.dst_fl = dst_fl;
        key.k = k_cycles; key.hgen = h->generation; key.sgen = s->generation;
        launches = enqueue_cycle(s, src_q, k_cycles, dst_qd, dst_qo, dst_fl, want_flags, n_chunks);
        if (launches < 0) return launches;
    }
    for (int k = 0; k < 3; ++k) VFK_CUDA(h, cudaStreamSynchronize(s->pipe[k]));
    return launches;
}

extern "C" int vfk_session_cycle(vfk_session s, const void* q_in, int k_cycles, void* qdot_out, void* q_out,
                                 int32_t* flags_out) {
    if (!s) return fail(nullptr, VFK_ERR_INVALID, "vfk_session_cycle: null session");
    vfk_ctx* h = s->h;
    if (k_cycles < 1) return fail(h, VFK_ERR_INVALID, "k_cycles must be >= 1");
    VFK_CUDA(h, cudaSetDevice(h->device));
    const size_t blk = (size_t)s->N * (size_t)s->n * s->es;
    char* pin_q = s->pin;
    char* pin_qd = s->pin + blk;
    char* pin_qo = s->pin + 2 * blk;
    char* pin_fl = s->pin + 3 * blk;
    // Caller buffers that are already page-locked are used directly; pageable ones go through the session's pinned staging
    // area.
    const char* src_q = nullptr;
    if (q_in) {
        src_q = (const char*)q_in;
        if (!host_pinned(q_in)) { memcpy(pin_q, q_in, blk); src_q = pin_q; }
    }
    const bool d_qd = qdot_out && host_pinned(qdot_out), d_qo = q_out && host_pinned(q_out), d_fl = flags_out && host_pinned(flags_out);
    char* dst_qd = qdot_out ? (d_qd ? (char*)qdot_out : pin_qd) : nullptr;
    char* dst_qo = q_out ? (d_qo ? (char*)q_out : pin_qo) : nullptr;
    char* dst_fl = flags_out ? (d_fl ? (char*)flags_out : pin_fl) : nullptr;
    const char* de = getenv("VFK_SESSION_DIRECT");
    const bool direct_ok = !(de && atoi(de) == 0) && q_in && s->n % 32 == 0 && s->n >= kDirectMinInstances;
    void *dq = nullptr, *dqd = nullptr;
    if (direct_ok) host_pinned(q_in, &dq);
    if (direct_ok && qdot_out) host_pinned(qdot_out, &dqd);
    const bool direct = dq && (!qdot_out || dqd) && ((uintptr_t)dq % 16 == 0) && ((uintptr_t)dqd % 16 == 0);
    const int launches = direct ? session_cycle_direct(s, dq, dqd, k_cycles, dst_qo, dst_fl, flags_out != nullptr)
                                : session_cycle_pipeline(s, src_q, k_cycles, dst_qd, dst_qo, dst_fl, flags_out != nullptr);
    if (launches < 0) return launches;
    if (qdot_out && !d_qd) memcpy(qdot_out, pin_qd, blk);
    if (q_out && !d_qo) memcpy(q_out, pin_qo, blk);
    if (flags_out && !d_fl) memcpy(flags_out, pin_fl, (size_t)s->n * 4);
    return launches;
}

extern "C" int vfk_session_solve(vfk_session s, const void* q_in, int max_cycles, double tol_trans, double tol_rot, void* q_out,
                                 int32_t* cycles_out, void* dist_out) {
    if (!s) return fail(nullptr, VFK_ERR_INVALID, "vfk_session_solve: null session");
    vfk_ctx* h = s->h;
    int rc;
    if (q_in && (rc = vfk_session_set_q(s, q_in)) != VFK_OK) return rc;
    vfk_buffers b;
    const int M = session_view(s, SessionOutputs::none, false, &b);
    if ((rc = vfk_solve(h, &b, s->n, M, max_cycles, tol_trans, tol_rot, (int32_t*)s->d_cycles, dist_out ? s->d_dist : nullptr, s->stream)) < 0)
        return rc;
    int launches = rc;
    char* stage = (char*)s->stage_out;                          // dense q [N][n], then dist [2][n]
    const size_t blk = (size_t)s->N * (size_t)s->n * s->es;
    if (q_out) {
        if ((rc = pack_dispatch(h, stage, b.q, s->N, 1, s->n, true, s->stream)) < 0) return rc;
        launches += rc;
        VFK_CUDA(h, cudaMemcpyAsync(q_out, stage, blk, cudaMemcpyDeviceToHost, s->stream));
    }
    if (dist_out) {
        if ((rc = pack_dispatch(h, stage + blk, s->d_dist, 2, 1, s->n, true, s->stream)) < 0) return rc;
        launches += rc;
        VFK_CUDA(h, cudaMemcpyAsync(dist_out, stage + blk, 2 * (size_t)s->n * s->es, cudaMemcpyDeviceToHost, s->stream));
    }
    if (cycles_out)         // one component: blocked == dense
        VFK_CUDA(h, cudaMemcpyAsync(cycles_out, s->d_cycles, (size_t)s->n * 4, cudaMemcpyDeviceToHost, s->stream));
    VFK_CUDA(h, cudaStreamSynchronize(s->stream));
    s->launches = launches;
    return launches;
}

extern "C" int vfk_session_enable(vfk_session s, const char* what, int on) {
    if (!s || !what) return fail(s ? s->h : nullptr, VFK_ERR_INVALID, "vfk_session_enable: null argument");
    bool* f = nullptr;
    if (!strcmp(what, "qdot_vf")) f = &s->en_vf;
    else if (!strcmp(what, "qdot_ns")) f = &s->en_ns;
    else if (!strcmp(what, "qdot_jp")) f = &s->en_jp;
    else if (!strcmp(what, "cmd")) f = &s->en_cmd;
    else if (!strcmp(what, "pose")) f = &s->en_pose;
    else if (!strcmp(what, "twist")) f = &s->en_twist;
    else return fail(s->h, VFK_ERR_INVALID, "vfk_session_enable: unknown output '%s'", what);
    *f = on != 0;
    s->generation++;
    return VFK_OK;
}

extern "C" int vfk_session_read(vfk_session s, const char* what, void* out) {
    if (!s || !what || !out) return fail(s ? s->h : nullptr, VFK_ERR_INVALID, "vfk_session_read: null argument");
    const void* src = nullptr;
    int rows = s->N;
    if (!strcmp(what, "qdot_vf")) src = s->b.qdot_vf;
    else if (!strcmp(what, "qdot_ns")) src = s->b.qdot_ns;
    else if (!strcmp(what, "qdot_jp")) src = s->b.qdot_jp;
    else if (!strcmp(what, "qdot")) src = s->b.qdot;
    else if (!strcmp(what, "cmd")) src = s->b.cmd;
    else if (!strcmp(what, "q")) src = s->b.q;
    else if (!strcmp(what, "jp_ref")) src = s->d_jp_ref;
    else if (!strcmp(what, "lastvec")) { src = s->b.ns_lastvec; rows = (ns_ctrl_vectors(s->N) > 0 ? ns_ctrl_vectors(s->N) : 1) * s->N; }
    else if (!strcmp(what, "pose")) { src = s->b.pose; rows = 12; }
    else if (!strcmp(what, "twist")) { src = s->b.twist; rows = 6; }
    else return fail(s->h, VFK_ERR_INVALID, "vfk_session_read: unknown field '%s'", what);
    vfk_ctx* h = s->h;
    VFK_CUDA(h, cudaSetDevice(h->device));
    int rc = pack_dispatch(h, s->stage_out, const_cast<void*>(src), rows, 1, s->n, true, s->stream);
    if (rc < 0) return rc;
    VFK_CUDA(h, cudaMemcpyAsync(out, s->stage_out, (size_t)rows * s->n * s->es, cudaMemcpyDeviceToHost, s->stream));
    VFK_CUDA(h, cudaStreamSynchronize(s->stream));
    return VFK_OK;
}

extern "C" int vfk_session_buffers(vfk_session s, vfk_buffers* out) {
    if (!s || !out) return fail(s ? s->h : nullptr, VFK_ERR_INVALID, "vfk_session_buffers: null argument");
    vfk_buffers v;
    session_view(s, SessionOutputs::all, true, &v);
    // the mixed-scene fields at the struct's end are written only in that mode: a caller built against the struct without
    // them never selects it, and its shorter struct is not written past its end
    memcpy(out, &v, s->obst_mode == VFK_OBST_MIXED ? sizeof v : offsetof(vfk_buffers, shared_obst));
    return VFK_OK;
}

// Releases whatever a (possibly half-built) session owns; every member starts null (value-initialised struct).
static void session_release(vfk_session_s* s) {
    cudaSetDevice(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    for (int k = 0; k < 3; ++k) if (s->pipe[k]) cudaStreamSynchronize(s->pipe[k]);
    if (s->pin) cudaFreeHost(s->pin);
    if (s->dev) cudaFree(s->dev);
    if (s->aux_dev) cudaFree(s->aux_dev);
    if (s->shared_dev) cudaFree(s->shared_dev);
    if (s->graph_exec) cudaGraphExecDestroy(s->graph_exec);
    if (s->stream) cudaStreamDestroy(s->stream);
    for (int k = 0; k < 3; ++k) if (s->pipe[k]) cudaStreamDestroy(s->pipe[k]);
    for (int k = 0; k < kMaxSessionChunks; ++k) {
        if (s->ev_up[k]) cudaEventDestroy(s->ev_up[k]);
        if (s->ev_done[k]) cudaEventDestroy(s->ev_done[k]);
    }
    if (s->ev_fork) cudaEventDestroy(s->ev_fork);
    for (int k = 0; k < 2; ++k) if (s->ev_join[k]) cudaEventDestroy(s->ev_join[k]);
    cudaGetLastError();
    delete s;
}

extern "C" void vfk_session_destroy(vfk_session s) {
    if (s) session_release(s);
}
