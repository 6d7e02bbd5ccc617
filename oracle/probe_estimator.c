/* Black-box probe of the reference's closed estimator block (state_output_step in src/libagilitycassie.a).  TEST INFRASTRUCTURE / study aid:
 * built by `make -C oracle probe` into oracle/_ref/libprobe_est.so (needs /root/reference); never shipped, never on the product path.
 * probe_est(in[45], ncalls, out[123]): in = motor pos[10] vel[10], joint pos[6] vel[6], IMU quat[4] gyro[3] accel[3], mag[3];
 * a fresh estimator is fed the same cassie_out `ncalls` times; out = state_out_t flattened as 123 doubles (field order of the struct). */
#include <string.h>
#include <stdlib.h>
#include "../include/cassie_bus.h"
typedef struct StateOutput state_output_t;
state_output_t *state_output_alloc(void); void state_output_setup(state_output_t *); void state_output_free(state_output_t *);
void state_output_step(state_output_t *, const cassie_out_t *, state_out_t *);
static elmo_out_t *drv(cassie_out_t *o, int i) { cassie_leg_out_t *l = i < 5 ? &o->leftLeg : &o->rightLeg; elmo_out_t *t[5] = {&l->hipRollDrive, &l->hipYawDrive, &l->hipPitchDrive, &l->kneeDrive, &l->footDrive}; return t[i % 5]; }
static cassie_joint_out_t *jnt(cassie_out_t *o, int i) { cassie_leg_out_t *l = i < 3 ? &o->leftLeg : &o->rightLeg; cassie_joint_out_t *t[3] = {&l->shinJoint, &l->tarsusJoint, &l->footJoint}; return t[i % 3]; }
static void fill(cassie_out_t *o, const double *in) {
  static const double tl[5] = {140.63, 140.63, 216.16, 216.16, 45.14}, gr[5] = {25, 25, 16, 16, 50};
  memset(o, 0, sizeof *o); o->isCalibrated = 1;
  o->pelvis.battery.dataGood = 1; o->pelvis.battery.stateOfCharge = 1;
  o->pelvis.radio.radioReceiverSignalGood = 1; o->pelvis.radio.receiverMedullaSignalGood = 1; o->pelvis.radio.channel[8] = 1;
  o->pelvis.vectorNav.dataGood = 1; o->pelvis.vectorNav.pressure = 101.325; o->pelvis.vectorNav.temperature = 25;
  for (int i = 0; i < 10; i++) { elmo_out_t *e = drv(o, i); e->statusWord = 0x0637; e->dcLinkVoltage = 48; e->driveTemperature = 30; e->torqueLimit = tl[i % 5]; e->gearRatio = gr[i % 5]; e->position = in[i]; e->velocity = in[10 + i]; }
  for (int i = 0; i < 6; i++) { jnt(o, i)->position = in[20 + i]; jnt(o, i)->velocity = in[26 + i]; }
  for (int k = 0; k < 4; k++) o->pelvis.vectorNav.orientation[k] = in[32 + k];
  for (int k = 0; k < 3; k++) { o->pelvis.vectorNav.angularVelocity[k] = in[36 + k]; o->pelvis.vectorNav.linearAcceleration[k] = in[39 + k]; o->pelvis.vectorNav.magneticField[k] = in[42 + k]; }
}
static void flat(const state_out_t *y, double *out) {
  int n = 0;
#define PUT(a, c) do { for (int k_ = 0; k_ < (c); k_++) out[n++] = (a)[k_]; } while (0)
  PUT(y->pelvis.position, 3); PUT(y->pelvis.orientation, 4); PUT(y->pelvis.rotationalVelocity, 3); PUT(y->pelvis.translationalVelocity, 3);
  PUT(y->pelvis.translationalAcceleration, 3); PUT(y->pelvis.externalMoment, 3); PUT(y->pelvis.externalForce, 3);            /* 0..21 */
  const state_foot_out_t *f[2] = {&y->leftFoot, &y->rightFoot};
  for (int s = 0; s < 2; s++) { PUT(f[s]->position, 3); PUT(f[s]->orientation, 4); PUT(f[s]->footRotationalVelocity, 3); PUT(f[s]->footTranslationalVelocity, 3); PUT(f[s]->toeForce, 3); PUT(f[s]->heelForce, 3); } /* 22..40, 41..59 */
  PUT(&y->terrain.height, 1); PUT(y->terrain.slope, 2);                                                                       /* 60..62 */
  PUT(y->motor.position, 10); PUT(y->motor.velocity, 10); PUT(y->motor.torque, 10); PUT(y->joint.position, 6); PUT(y->joint.velocity, 6); /* 63..104 */
  (void)n;
}
void probe_est(const double *in, int ncalls, double *out) {
  cassie_out_t o; state_out_t y; fill(&o, in);
  state_output_t *e = state_output_alloc(); state_output_setup(e);
  for (int i = 0; i < ncalls; i++) state_output_step(e, &o, &y);
  flat(&y, out); state_output_free(e);
}
/* a sequence: T inputs of 45, one persistent estimator, T outputs of 105 */
void probe_est_seq(const double *in, int T, double *out) {
  cassie_out_t o; state_out_t y;
  state_output_t *e = state_output_alloc(); state_output_setup(e);
  for (int t = 0; t < T; t++) { fill(&o, in + 45 * t); state_output_step(e, &o, &y); flat(&y, out + 105 * t); }
  state_output_free(e);
}

/* pd_input_step probe: in[45] as above (cassie_out), task[60] = left-leg taskPd {torque, pTarget, dTarget, pGain, dGain}[6] then the right leg's;
 * out[10] = cassie_user_in_t.torque after ncalls calls on a fresh block */
typedef struct PdInput pd_input_t;
pd_input_t *pd_input_alloc(void); void pd_input_setup(pd_input_t *); void pd_input_free(pd_input_t *);
void pd_input_step(pd_input_t *, const pd_in_t *, const cassie_out_t *, cassie_user_in_t *);
void probe_pd(const double *in, const double *task, int ncalls, double *out) {
  cassie_out_t o; fill(&o, in);
  pd_in_t u; memset(&u, 0, sizeof u);
  for (int s = 0; s < 2; s++) { pd_task_in_t *t = s ? &u.rightLeg.taskPd : &u.leftLeg.taskPd; const double *p = task + 30 * s;
    for (int k = 0; k < 6; k++) { t->torque[k] = p[k]; t->pTarget[k] = p[6 + k]; t->dTarget[k] = p[12 + k]; t->pGain[k] = p[18 + k]; t->dGain[k] = p[24 + k]; } }
  cassie_user_in_t ui; memset(&ui, 0, sizeof ui);
  pd_input_t *pd = pd_input_alloc(); pd_input_setup(pd);
  for (int i = 0; i < ncalls; i++) pd_input_step(pd, &u, &o, &ui);
  for (int i = 0; i < 10; i++) out[i] = ui.torque[i];
  pd_input_free(pd);
}

/* cassie_core_sim_step probe: in[45] (cassie_out), u[10] commanded torques, radio channel 8 -> out[10] torques of cassie_in_t */
typedef struct CassieCoreSim cassie_core_sim_t;
cassie_core_sim_t *cassie_core_sim_alloc(void); void cassie_core_sim_setup(cassie_core_sim_t *); void cassie_core_sim_free(cassie_core_sim_t *);
void cassie_core_sim_step(cassie_core_sim_t *, const cassie_user_in_t *, const cassie_out_t *, cassie_in_t *);
void probe_core(const double *in, const double *u, double ch8, double *out) {
  cassie_out_t o; fill(&o, in); o.pelvis.radio.channel[8] = ch8;
  cassie_user_in_t ui; memset(&ui, 0, sizeof ui); for (int i = 0; i < 10; i++) ui.torque[i] = u[i];
  cassie_in_t ci; memset(&ci, 0, sizeof ci);
  cassie_core_sim_t *c = cassie_core_sim_alloc(); cassie_core_sim_setup(c);
  cassie_core_sim_step(c, &ui, &o, &ci);
  for (int i = 0; i < 10; i++) { const cassie_leg_in_t *l = i < 5 ? &ci.leftLeg : &ci.rightLeg; const elmo_in_t *t[5] = {&l->hipRollDrive, &l->hipYawDrive, &l->hipPitchDrive, &l->kneeDrive, &l->footDrive}; out[i] = t[i % 5]->torque; }
  cassie_core_sim_free(c);
}

/* the chain oracle/fuzz_agility.c checks, on fresh blocks: in[45] (cassie_out), a whole pd_in_t, radio channel 8 -> pd[10] = cassie_user_in_t.torque
 * of pd_input_step, core[10] = the drive torques cassie_core_sim_step makes of them */
void probe_pd_core(const double *in, const pd_in_t *u, double ch8, double *pd, double *core) {
  cassie_out_t o; fill(&o, in); o.pelvis.radio.channel[8] = ch8;
  cassie_user_in_t ui; memset(&ui, 0, sizeof ui);
  pd_input_t *p = pd_input_alloc(); pd_input_setup(p); pd_input_step(p, u, &o, &ui); pd_input_free(p);
  for (int i = 0; i < 10; i++) pd[i] = ui.torque[i];
  cassie_in_t ci; memset(&ci, 0, sizeof ci);
  cassie_core_sim_t *c = cassie_core_sim_alloc(); cassie_core_sim_setup(c); cassie_core_sim_step(c, &ui, &o, &ci); cassie_core_sim_free(c);
  for (int i = 0; i < 10; i++) { const cassie_leg_in_t *l = i < 5 ? &ci.leftLeg : &ci.rightLeg; const elmo_in_t *t[5] = {&l->hipRollDrive, &l->hipYawDrive, &l->hipPitchDrive, &l->kneeDrive, &l->footDrive}; core[i] = t[i % 5]->torque; }
}

/* as probe_est, plus the drives' measured torques: in[45..54] */
void probe_est_tq(const double *in, int ncalls, double *out) {
  cassie_out_t o; state_out_t y; fill(&o, in);
  for (int i = 0; i < 10; i++) drv(&o, i)->torque = in[45 + i];
  state_output_t *e = state_output_alloc(); state_output_setup(e);
  for (int i = 0; i < ncalls; i++) state_output_step(e, &o, &y);
  flat(&y, out); state_output_free(e);
}

/* internal-memory view of the estimator (study aid): T inputs of 45, one persistent block; mem = T+1 snapshots (after setup, then after each call)
 * of the first `nbytes` bytes of the block; returns malloc_usable_size of the block. */
#include <malloc.h>
long probe_est_mem(const double *in, int T, unsigned char *mem, long nbytes, double *out) {
  cassie_out_t o; state_out_t y;
  state_output_t *e = state_output_alloc(); state_output_setup(e);
  long sz = (long)malloc_usable_size(e);
  if (nbytes > sz) nbytes = sz;
  if (mem) memcpy(mem, e, nbytes);
  for (int t = 0; t < T; t++) { fill(&o, in + 45 * t); state_output_step(e, &o, &y); if (out) flat(&y, out + 105 * t); if (mem) memcpy(mem + (t + 1) * nbytes, e, nbytes); }
  state_output_free(e);
  return sz;
}
/* same with raw cassie_out_t records (T of them, as the simulator wrote them) */
long probe_est_mem_raw(const cassie_out_t *seq, int T, unsigned char *mem, long nbytes, double *out) {
  state_out_t y;
  state_output_t *e = state_output_alloc(); state_output_setup(e);
  long sz = (long)malloc_usable_size(e);
  if (nbytes > sz) nbytes = sz;
  if (mem) memcpy(mem, e, nbytes);
  for (int t = 0; t < T; t++) { state_output_step(e, seq + t, &y); if (out) flat(&y, out + 105 * t); if (mem) memcpy(mem + (t + 1) * nbytes, e, nbytes); }
  state_output_free(e);
  return sz;
}
/* does state_output_setup on a used block restart the filters?  out[0..104] = output of a call after `pre` calls + setup; out[105..209] = same from a fresh block */
void probe_est_resetup(const double *in, int pre, double *out) {
  cassie_out_t o; state_out_t y; fill(&o, in);
  state_output_t *e = state_output_alloc(); state_output_setup(e);
  for (int i = 0; i < pre; i++) state_output_step(e, &o, &y);
  state_output_setup(e); state_output_step(e, &o, &y); flat(&y, out); state_output_free(e);
  e = state_output_alloc(); state_output_setup(e); state_output_step(e, &o, &y); flat(&y, out + 105); state_output_free(e);
}
