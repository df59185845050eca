// b2_types.h — device-side model / data / shared-memory layout descriptors (internal).
#pragma once
#include <stdint.h>

#ifndef B2_WARPS_PER_CTA
#define B2_WARPS_PER_CTA 4
#endif
#ifndef B2_MIN_CTAS
// 16 warps per SM: the kernel fits 128 registers without spills (ptxas only takes more when allowed to), and the
// per-environment shared-memory block of the G1 scene (13.1 KB at 35 contacts) lets four 4-warp CTAs share an SM
#define B2_MIN_CTAS (16 / B2_WARPS_PER_CTA)
#endif
#define B2_MAX_FIELDS 96

enum { JNT_FREE = 0, JNT_BALL = 1, JNT_SLIDE = 2, JNT_HINGE = 3 };
#define GP 15  // shared-memory collision pose records: pos[3], mat[9], rbound, margin (+1 pad: odd stride)
enum { G_PLANE = 0, G_HFIELD = 1, G_SPHERE = 2, G_CAPSULE = 3, G_ELLIPSOID = 4, G_CYLINDER = 5, G_BOX = 6, G_MESH = 7 };
enum { OBJ_BODY = 1, OBJ_XBODY = 2, OBJ_GEOM = 5 };
enum { INT_EULER = 0, INT_IMPLICITFAST = 3 };
enum { SOL_PGS_ = 0, SOL_CG_ = 1, SOL_NEWTON_ = 2 };

// The float model arrays a caller may expand per world, in DevModel's member order:
// X(name, trailing width of the caller's view, element count in model sizes).  Width 1 is a 1-D view per world.
#define B2_MODEL_FARRAYS(X)                                                                                       \
  X(body_pos, 3, nbody) X(body_quat, 4, nbody) X(body_ipos, 3, nbody) X(body_iquat, 4, nbody)                    \
  X(body_mass, 1, nbody) X(body_subtreemass, 1, nbody) X(body_inertia, 3, nbody) X(body_invweight0, 2, nbody)    \
  X(jnt_pos, 3, njnt) X(jnt_axis, 3, njnt) X(jnt_range, 2, njnt) X(jnt_solref, 2, njnt) X(jnt_solimp, 5, njnt)   \
  X(jnt_margin, 1, njnt) X(jnt_stiffness, 1, njnt)                                                               \
  X(dof_armature, 1, nv) X(dof_damping, 1, nv) X(dof_frictionloss, 1, nv) X(dof_invweight0, 1, nv)               \
  X(geom_size, 3, ngeom) X(geom_pos, 3, ngeom) X(geom_quat, 4, ngeom) X(geom_friction, 3, ngeom)                 \
  X(geom_solref, 2, ngeom) X(geom_solimp, 5, ngeom) X(geom_solmix, 1, ngeom) X(geom_margin, 1, ngeom)            \
  X(geom_gap, 1, ngeom) X(geom_rbound, 1, ngeom) X(geom_rgba, 4, ngeom) X(site_pos, 3, nsite)                    \
  X(site_quat, 4, nsite) X(actuator_gainprm, 10, nu) X(actuator_biasprm, 10, nu) X(actuator_ctrlrange, 2, nu)    \
  X(actuator_forcerange, 2, nu) X(actuator_gear, 1, nu) X(qpos0, 1, nq)

// A float model array; `stride` is the per-world stride in floats (0 = shared by all worlds).
struct FArr {
  const float* p;
  int stride;
  int n;
};

// Per-world Data array: base pointer + row stride in elements (rows padded to 16 B).
struct DArr {
  float* p;
  int stride;
  int n;
};
struct IArr {
  int* p;
  int stride;
  int n;
};

// Per-contact SoA fields inside the per-env shared-memory block (index f*maxcon + c).
enum {
  CS0 = 0,        // 18 floats: S_m[a] at CS0 + m*6 + a; S_m = [r x e_m ; e_m], e_0 = normal
  CDIST = 18, CMU, CD, CKI, CB,
  CINFO,  // int: body1 | body2 << 8 | condim << 16 | active rows << 20 | body-pair group << 24
  CJAR0, CJAR1, CJAR2, CJAR3,
  CJV0, CJV1, CJV2, CJV3,
  C_NFIELD  // 32
};
// Per-limit-row SoA fields (index f*nlimcap + r).
enum { LINFO = 0, LD, LJAR, LJV, L_NFIELD };

// Offsets (in floats) of every region of one environment's shared-memory block.
struct Layout {
  int total;  // floats per env (multiple of 4)
  // bulk-loaded inputs (16 B aligned)
  int qpos, qvel, qacc_ws;  // (ctrl, qfrc_applied and xfrc_applied have one use each and are read from global memory)
  // kinematics
  int xpos, xquat, xipos, scom, xanchor, xaxis;
  // smooth dynamics
  int cinert, crb, cdof, cdofdot, cvel, cacc;
  int H, invdiag;  // (the joint-space inertia M itself lives in global memory: Data field qM_packed)
  int qfrc_smooth, qacc_smooth, qacc, Ma, grad, search, Mv, qfrc_c, tmpv, actf;
  // collision / constraints (overlaid on smooth-only regions)
  int gpose, pairlist, contacts, limits, gstart, gV, glist, gA, gu, gW;
  int sens;
  int Mred;   // Schur complement of M on the leading ndcap x ndcap block (reduced Newton problem)
  int ndcap;  // largest leading block the reduced solver may use (nv - 4k, packed size <= the Mred region)
  int maxcon, nlimcap, maxpair;
};

struct DevModel {
  int nq, nv, nu, nbody, njnt, ngeom, nsite, nsensor, nsensordata, npair, ncg, maxdepth;
  int ntri;  // nv*(nv+1)/2
  int maxcon, njmax;
  int integrator, iterations, ls_iterations, solver;
  int debug;  // test hooks: 1 debug outputs, 2 dense LDL schedule, 4 Newton on all dofs
  float timestep, tolerance, ls_tolerance, impratio, meaninertia;
  float gravity[3];
  // integer tables
  const int *body_parentid, *body_rootid, *body_jntadr, *body_jntnum, *body_dofadr, *body_dofnum;
  const int *body_chain, *body_depth;
  const unsigned long long *body_dofmask, *body_ancmask;
  const unsigned long long *body_submask, *dof_bodymask;  // descendants of a body / bodies moved by a dof
  const float4* kinrec;  // 4 x float4 per body: compact kinematic record (valid when fastkin)
  int fastkin;
  const int *jnt_type, *jnt_qposadr, *jnt_dofadr, *jnt_bodyid, *jnt_limited;
  const int *dof_bodyid, *dof_jntid, *dof_parentid;
  const int *geom_type, *geom_bodyid, *geom_condim, *geom_priority, *geom_cslot, *cgeom;
  const int *site_bodyid;
  const int *actuator_trnid, *actuator_ctrllimited, *actuator_forcelimited;
  const int *pair_geom1, *pair_geom2;
  // height-field pairs, grouped by field (hierarchical broadphase; all nullptr / 0 without fields):
  int nhf, nhfd, n_nhpair;    // distinct fields, distinct geoms paired with a field, pairs without a field
  const int* hfl_slot;        // [nhf] pose slot of the field (or -2 - index into fixed_pose)
  const int* hfl_geom;        // [nhf] its geom id
  const float4* hfl_box;      // [nhf] its box (rx, ry, elevation, base)
  const int* hfl_start;       // [nhf + 1] range of the field's pairs in hfl_pairs
  const int* hfl_pairs;       // pair indices, ascending per field
  const int* hfd_slot;        // [nhfd] pose slots of the geoms paired with a field
  const int* nh_pairs;        // [n_nhpair] indices of the pairs without a field, ascending (nullptr: all pairs)
  const unsigned* pair_word;  // broadphase record per pair: slot1 | slot2 << 12 | (geom1 is a height field) << 30 | (geom1 is a plane) << 31
  // grid-static collision set (terrain): geoms welded to the world, found through a uniform xy grid
  int nstatic, ndyn, nposegeom, grid_nx, grid_ny;
  float grid_x0, grid_y0, grid_cell;
  const int *geom_contype, *geom_conaffinity;
  const int *posegeom;     // geoms whose world pose is recomputed every step (all but the grid-static ones)
  const int *dyn_cgeom;    // dynamic collision geoms that visit the grid
  const int *static_geom, *static_cell0, *grid_start, *grid_items;
  const float* static_pose;  // 16 floats per static geom: pos[3], mat[9], rbound, pad[3] (world 0's model values)
  int nfixed;                // height fields welded to the world: posed once at create, no shared-memory pose slot
  const float* fixed_pose;   // [nfixed][16], same record as static_pose
  const int* fixed_geom;     // [nfixed] geom ids
  // mesh / height-field assets (b2_convex.h): geom_dataid -> mesh or hfield id; shared by all worlds
  const int *geom_dataid, *mesh_vertadr, *mesh_vertnum, *hfield_adr, *hfield_nrow, *hfield_ncol;
  const float *mesh_vert, *hfield_size, *hfield_data;
  const int *sensor_objtype, *sensor_objid, *sensor_reftype, *sensor_refid, *sensor_intprm;
  const int *sensor_adr, *sensor_dim;
  // bottom-up (leaves first) blocked L^T D L: trailing-update schedules, one word per target entry
  // p | i << 12 | j << 18.  ldl_dense: every packed index in order (a block with m leading rows uses the
  // first tri(m)); ldl_sparse: per block only the entries the dof tree can make non-zero.
  const unsigned *ldl_dense, *ldl_sparse;
  int ldl_start[18];
  int ldl_nsparse;
  // float arrays (expandable per world)
#define B2_FARR_MEMBER(name, width, count) FArr name;
  B2_MODEL_FARRAYS(B2_FARR_MEMBER)
#undef B2_FARR_MEMBER
  Layout lay;
};

struct DevData {
  int nworld;
  int world_base, world_count;  // this launch covers launch slots [0, world_count) -> worlds from world_base
  DArr qpos, qvel, ctrl, qacc_warmstart, qfrc_applied, xfrc_applied, act;
  DArr qacc, xpos, xquat, xmat, xipos, subtree_com, cvel, geom_xpos, geom_xmat, site_xpos,
      site_xmat, sensordata, actuator_force, time;
  DArr qacc_smooth_prev, ctrl_prev;  // previous step's unconstrained acceleration and control (shifted warm start)
  DArr qM_packed;  // joint-space inertia, packed lower triangle (engine scratch between phases; L2-resident)
  DArr link_vel_w, com_vel_w, link_state_b;  // per body: EntityData's derived velocities / body-frame state
  DArr qfrc_bias, qfrc_smooth, qacc_smooth, qfrc_constraint, qM;
  DArr contact_dist, contact_pos, contact_frame, contact_force, solver_cost;
  IArr ncon, nefc, solver_niter, contact_geom, overflow, solver_nd, solver_nls;
  int emit;                         // write consumer-visible kinematics (0 for all but the last sub-step of a decimation loop)
  int phase_sync;                   // CTA barriers at phase boundaries (every warp of the launch owns an environment)
  const int* world_order;           // optional: launch slot -> world (heavy-first dispatch)
  const unsigned char* world_mask;  // optional: worlds with mask 0 are skipped (masked forward)
};
