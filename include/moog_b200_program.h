/*
 * moog_b200_program.h -- binary layout of a compiled MOOG task ("program") and
 * of the per-env state record the kernels operate on.
 *
 * A *program* is what the host-side config compiler produces from the dict a
 * MOOG config's get_config(level) returns (reference:
 * moog/environment.py:28-35 -- state_initializer, physics, task, action_space,
 * observers, game_rules).  It is a flat, position-independent blob:
 *
 *     int32   hdr[MOOG_HDR_WORDS]
 *     moog_op ops[hdr[MOOG_H_N_OPS]]
 *     int32   ipool[hdr[MOOG_H_N_IPOOL]]      (padded to a multiple of 2)
 *     moog_ex expr[hdr[MOOG_H_N_EXPR]]
 *     double  dpool[hdr[MOOG_H_N_DPOOL]]      (shape table and sampler parameters of the
 *                                              device-side reset sampler; may be empty)
 *
 * Sections of `ops` (forces, correctives, rules, tasks, actions, conditions)
 * are addressed by (start, count) pairs in the header.  Layer lists live in
 * `ipool`; small per-sprite predicates / assignments (the lambdas MOOG configs
 * pass as filters, conditions and modifiers) are postfix programs in `expr`.
 *
 * State of env n (all arrays owned by the caller; N envs, S sprite slots,
 * L layers; slots of layer l are [layer_off[l], layer_off[l+1]) and the live
 * sprites of a layer are its first cnt[n][l] slots, in MOOG list order, which
 * is also z-order -- reference moog/environment.py:20-25):
 *
 *     double  dyn [N][MOOG_DYN_FIELDS ][S]   x y vx vy angle angle_vel
 *     double  stat[N][MOOG_STAT_FIELDS][S]   mass scale aspect ix iy max_radius c0 c1 c2 opacity
 *     int32   meta[N][MOOG_META_FIELDS][S]   shape_id flags n_vertices
 *     double  vtx [N][VT][2]                 cached WORLD vertices; slot s owns
 *                                            vertices [voff[s], voff[s]+nv)
 *     int32   cnt [N][MOOG_MAX_LAYERS]
 *     int32   envi[N][MOOG_ENVI_WORDS]       step_count reset_next err episodes rng...
 *     double  envf[N][hdr[MOOG_H_N_ENVF]]    action-space memory, task countdowns
 *
 * `vtx` mirrors the reference's Sprite._path cache (moog/sprite.py:411-424):
 * the reference never recomputes world vertices from (position, angle, scale)
 * during an episode, it translates / rotates the cached path incrementally
 * (sprite.py:531-540, 616-633).  The roundings of that cache decide exact
 * ties -- two identical circles colliding head-on pick the contact side by the
 * last bit -- so the cache is state, not a derived quantity.
 *
 * The per-env record is contiguous and field-major so that a warp that owns
 * one env reads it with unit-stride, fully coalesced loads (lane == slot).
 */
#ifndef MOOG_B200_PROGRAM_H_
#define MOOG_B200_PROGRAM_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MOOG_MAGIC 0x474F4F4D /* "MOOG" little endian */
#define MOOG_VERSION 1

#define MOOG_MAX_LAYERS 16
#define MOOG_MAX_VERTS 32   /* per sprite that takes part in overlap tests / collisions (lane = vertex);
                               'circle' is a 30-gon (moog/shapes.py:17) */
#define MOOG_MAX_OUTLINE 128 /* per sprite that is only moved and drawn (e.g. the 102-vertex annulus occluder of
                               the first-person configs, shapes.py:170-188) */
#define MOOG_MAX_SLOTS 256

#define MOOG_DYN_FIELDS 6
enum { MOOG_D_X = 0, MOOG_D_Y, MOOG_D_VX, MOOG_D_VY, MOOG_D_ANG, MOOG_D_ANGVEL };

#define MOOG_STAT_FIELDS 10
enum {
  MOOG_S_MASS = 0, MOOG_S_SCALE, MOOG_S_ASPECT, MOOG_S_IX, MOOG_S_IY,
  MOOG_S_MAXR, MOOG_S_C0, MOOG_S_C1, MOOG_S_C2, MOOG_S_OPACITY
};

#define MOOG_META_FIELDS 3
enum { MOOG_M_SHAPE = 0, MOOG_M_FLAGS, MOOG_M_NV };
#define MOOG_SF_CIRCLE 1 /* shape name == 'circle' (moog/sprite.py:500-502) */
/* NumPy dtype of the reference's per-sprite fields (SURVEY fact 10): a sampled
 * velocity is a float32 ndarray, a sampled angle_vel a float32 0-d array, and
 * the angle turns float32 with it.  kind: 0 python float, 1 float32, 2 float64. */
#define MOOG_SF_VEL32 2
#define MOOG_SF_TELEPORTING 64 /* Portal._currently_teleporting holds this sprite's id (portal.py:61-76) */
#define MOOG_SF_ANGVEL_SHIFT 2 /* 2 bits */
#define MOOG_SF_ANG_SHIFT 4    /* 2 bits */
/* Velocity-array aliasing.  `Tether(update_angle_vel=False)` assigns ONE ndarray
 * object to every tethered sprite (`s.velocity = total_velocity`,
 * tether_physics.py:86-91; the setter keeps the object, sprite.py:639-643), so a
 * later in-place `sprite.velocity += dv` of any force (abstract_force.py:64-74,
 * collisions.py) changes all of them.  The reference's own tether known-answer
 * test depends on it.  Sprites whose flags carry the same non-zero alias id share
 * their velocity; an assignment (`sprite.velocity = v`) clears the id. */
#define MOOG_SF_VALIAS_SHIFT 8 /* 23 bits */
#define MOOG_SF_VALIAS_MASK 0x7fffff

#define MOOG_ENVI_WORDS 8
enum {
  MOOG_EI_STEP_COUNT = 0, MOOG_EI_RESET_NEXT, MOOG_EI_ERR, MOOG_EI_EPISODES,
  MOOG_EI_CREATED,      /* CreateSprites calls this env has made (keys their Philox draws) */
  MOOG_EI_RULE_PASSES,  /* passes over the game rules this env has made (keys the rule-noise draws) */
  MOOG_EI_LAST_RESET, MOOG_EI_VALIAS_NEXT /* last alias id handed out */
};

/* error bits (data-dependent reference exceptions, raised lazily by the host) */
#define MOOG_ERR_NORMAL_NOT_UNIT 1u  /* collisions.py:323-326 ValueError        */
#define MOOG_ERR_DISJOINT_LOOP   2u  /* collisions.py:740 loop would not end     */
#define MOOG_ERR_TETHER_ZIP      4u  /* tether_physics.py:192-196 ValueError     */
#define MOOG_ERR_LAYER_OVERFLOW  8u  /* layer capacity exceeded                  */
#define MOOG_ERR_OFF_MAZE_GRID   16u /* maze_physics.py:93-104 ValueError (sprite not on the maze grid) */

/* header words */
#define MOOG_HDR_WORDS 64
enum {
  MOOG_H_MAGIC = 0, MOOG_H_VERSION, MOOG_H_BYTES, MOOG_H_N_LAYERS, MOOG_H_N_SLOTS,
  MOOG_H_K, MOOG_H_N_OPS, MOOG_H_N_IPOOL, MOOG_H_N_EXPR, MOOG_H_N_ENVF,
  MOOG_H_FORCES, MOOG_H_N_FORCES, MOOG_H_CORR, MOOG_H_N_CORR,
  MOOG_H_RULES, MOOG_H_N_RULES, MOOG_H_TASKS, MOOG_H_N_TASKS,
  MOOG_H_ACTIONS, MOOG_H_N_ACTIONS, MOOG_H_ACTION_DIM, MOOG_H_NOISE_DIM,
  MOOG_H_R_HEIGHT, MOOG_H_R_WIDTH, MOOG_H_R_AA, MOOG_H_R_BG, /* bg = r | g<<8 | b<<16 */
  MOOG_H_R_COLORMAP, MOOG_H_R_MODIFIER, MOOG_H_R_MOD_LAYER, MOOG_H_R_ENABLED,
  MOOG_H_RULE_NOISE_DIM, /* uniforms per env per step consumed by sample_one rules */
  MOOG_H_VOFF,           /* index in ipool of voff[S+1]: first cached vertex of each slot */
  MOOG_H_LAYER_OFF = 32, /* MOOG_MAX_LAYERS+1 words */
  MOOG_H_N_VTX = 49,     /* VT: cached vertices per env */
  MOOG_H_RESET = 51,      /* first MOOG_Z_* op of the device-side reset sampler */
  MOOG_H_N_RESET = 52,    /* number of them (0: resets draw from the caller's pool only) */
  MOOG_H_N_DPOOL = 53,    /* doubles in dpool */
  MOOG_H_SHAPE_TAB = 54,  /* index in ipool of shape_off[n_shapes]: offset in dpool of each shape record */
  MOOG_H_N_META = 55,     /* numeric `sprite.metadata[key]` columns the program's callables read (<= MOOG_MAX_META) */
  MOOG_H_N_METAVAR = 57,  /* entries of the env's `meta_state` dict carried in envf (numbers; strings as codes) */
  MOOG_H_METAVAR_OFF = 58,  /* envf offset of the first one */
  MOOG_H_METAVAR_INIT = 59, /* dpool index of their values after meta_state_initializer() (environment.py:86) */
  MOOG_H_VIEWS = 60,      /* index in ipool of the view table: MOOG_H_N_VIEWS rows of MOOG_VIEW_WORDS */
  MOOG_H_N_VIEWS = 61,    /* PILRenderer observers after the first (views 1..); 0 = one renderer or none */
  MOOG_H_MASKS = 62,      /* index in ipool of the mask table: MOOG_H_N_MASKS rows of MOOG_VIEW_WORDS */
  MOOG_H_N_MASKS = 63,    /* SpriteMask observers (0 = none, and no table) */
  MOOG_H_META_OFF = 56,   /* envf offset of column 0; column k of slot s is envf[off + k * S + s], NaN = no such key.
                             Read as attribute MOOG_AT_META0 + k; travels with the sprite when slots are compacted */
  MOOG_H_CMASK_WORDS = 50 /* 32-bit words of the per-env broad-phase candidate matrices of all
                             MOOG_F_COLLISION ops (rows = capacity of layer a, ceil(capacity of
                             layer b / 32) words per row).  Derived: moog_program_create fills
                             it in, whatever the blob says. */
};

/* Views: one per PILRenderer observer, in the order of the config's observers dict.  View 0's settings
 * are the header words MOOG_H_R_HEIGHT .. MOOG_H_R_ENABLED; view k >= 1 is row k - 1 of the view table,
 * ipool[hdr[MOOG_H_VIEWS] + MOOG_VIEW_WORDS * (k - 1) ...], whose words are in the same order.  The
 * renderer reads every view through a pointer to its MOOG_VIEW_WORDS words. */
#define MOOG_VIEW_WORDS 8
#define MOOG_MAX_VIEWS 8 /* renderers per program, view 0 included */
enum {
  MOOG_V_HEIGHT = 0, MOOG_V_WIDTH, MOOG_V_AA, MOOG_V_BG, MOOG_V_COLORMAP, MOOG_V_MODIFIER, MOOG_V_MOD_LAYER,
  MOOG_V_ENABLED
};
#ifdef __cplusplus
#define MOOG_STATIC_ASSERT_ static_assert
#else
#define MOOG_STATIC_ASSERT_ _Static_assert
#endif
MOOG_STATIC_ASSERT_(MOOG_H_R_WIDTH - MOOG_H_R_HEIGHT == MOOG_V_WIDTH && MOOG_H_R_AA - MOOG_H_R_HEIGHT == MOOG_V_AA &&
                        MOOG_H_R_BG - MOOG_H_R_HEIGHT == MOOG_V_BG &&
                        MOOG_H_R_COLORMAP - MOOG_H_R_HEIGHT == MOOG_V_COLORMAP &&
                        MOOG_H_R_MODIFIER - MOOG_H_R_HEIGHT == MOOG_V_MODIFIER &&
                        MOOG_H_R_MOD_LAYER - MOOG_H_R_HEIGHT == MOOG_V_MOD_LAYER &&
                        MOOG_H_R_ENABLED - MOOG_H_R_HEIGHT == MOOG_V_ENABLED && MOOG_V_ENABLED + 1 == MOOG_VIEW_WORDS,
                    "the header's renderer words are a view row");
#undef MOOG_STATIC_ASSERT_

/* Masks: one per SpriteMask observer, in the order of the config's observers dict, independent of the
 * views (a program may have masks and no renderer).  Mask k is row k of the mask table,
 * ipool[hdr[MOOG_H_MASKS] + MOOG_VIEW_WORDS * k ...], in view-row order: MOOG_V_AA = 1, MOOG_V_BG = 0,
 * MOOG_V_COLORMAP = 0, MOOG_V_MODIFIER / MOOG_V_MOD_LAYER as for a renderer, MOOG_V_ENABLED = 1.  At most
 * MOOG_MAX_VIEWS masks.  A mask is int16 mask[N][H][W]: the slot of the last sprite in draw order whose
 * Pillow polygon fill covers the pixel (row 0 = top, as the frames), -1 where none does; sprites whose
 * ink alpha byte is 0 are not drawn. */

enum { MOOG_CMAP_NONE = 0, MOOG_CMAP_HSV = 1 };
enum { MOOG_PMOD_NONE = 0, MOOG_PMOD_FIRST_PERSON = 1, MOOG_PMOD_TORUS = 2 };

typedef struct {
  int32_t kind;
  int32_t flags;
  int32_t i[6];
  double p[6];
} moog_op; /* 80 bytes */

/* op kinds ---------------------------------------------------------------- */
enum {
  /* forces: i[0]=layer a, i[1]=layer b (-1 if unary) */
  MOOG_F_DRAG = 1,          /* p0 coeff            friction.py:54-56          */
  MOOG_F_KINETIC_FRICTION,  /* p0 coeff            friction.py:25-33          */
  MOOG_F_DOWN_GRAVITY,      /* p0 g                gravity.py:21-23           */
  MOOG_F_GRAVITY,           /* p0 g, SYMMETRIC     gravity.py:44-60           */
  MOOG_F_RANDOM,            /* p0 max magnitude; i[2] noise column  random_force.py:22-26 */
  MOOG_F_DIST_LINEAR,       /* p0 intercept p1 slope p2 horizon  distance_fn_force.py:48-74 */
  MOOG_F_DIST_SPRING,       /* p0 k p1 equilibrium distance_fn_force.py:77-89 */
  MOOG_F_COLLISION,         /* p0 elasticity; i[2] max_recursion  collisions.py:494-584 */
  MOOG_F_MAZE_WALK,         /* RandomMazeWalk: p0 speed; i[2] noise column (4 per sprite of the layer's
                               capacity: np.random.rand(2, 2)); i[3] envf offset of the maze record;
                               flags PREVENT_BACKTRACKING / ALLOW_WALL_BACKTRACKING / ONLY_TURN_AT_WALL
                               maze_walk.py:97-196 */

  /* corrective physics: i[0]=ipool start of layer list, i[1]=count */
  MOOG_C_TETHER = 32,       /* p0,p1 anchor        tether_physics.py:126-140  */
  MOOG_C_TETHER_ZIPPED,     /*                     tether_physics.py:186-201  */
  MOOG_C_CONSTANT_SPEED,    /* p0 speed            constant_speed.py:34-46    */
  MOOG_C_MAZE_PHYSICS,      /* i0,i1 avatar layer list; i[2] envf offset of the maze record; p0 constant_speed,
                               p1 max_speed (NaN = None)   maze_physics.py:19-211 */

  /* rules */
  MOOG_R_VANISH_ON_CONTACT = 64, /* i0 vanishing layer, i1 contacting layer  vanish.py:66-86 */
  MOOG_R_VANISH_BY_FILTER,       /* i0 layer, i2 filter expr (-1: all)       vanish.py:42-63 */
  MOOG_R_MODIFY_ON_CONTACT,      /* i0,i1 list0; i2,i3 list1; i4 -> ipool[4]: mod0 filt0 mod1 filt1  contact_rules.py:54-120 */
  MOOG_R_MODIFY_SPRITES,         /* i0,i1 list; i2 modifier, i3 filter; SAMPLE_ONE; i4 noise column  modify_sprites.py:35-52 */
  MOOG_R_COND_BEGIN,             /* i0 condition op index, i1 number of following rule ops guarded   conditional.py:55-58 */
  MOOG_R_TIMED_BEGIN,            /* TimedRule / DelayedRule / TemporaryRule: i1 number of following rule ops guarded,
                                    i2 envf slot of (steps_until_start, steps_until_stop), p0,p1 the interval
                                    they are reset to                                                   timing.py:15-107 */
  MOOG_R_KEEP_NEAR_CENTER,       /* i0 agent layer, i1,i2 list of the layers to move, p0,p1 grid cell    re_center.py:13-76 */
  MOOG_R_PORTAL,                 /* i0 teleporting layer, i1 portal layer (paired in order); a sprite that has
                                    teleported carries MOOG_SF_TELEPORTING until it is in no portal       portal.py:41-76 */
  MOOG_R_CHANGE_LAYER,           /* i0 old layer, i1 new layer, i2 filter expr (-1: all): the flagged sprites
                                    are appended to the new layer in order and popped from the old one
                                                                                                 change_layer.py:34-45 */
  MOOG_R_CREATE_SPRITES,         /* create_sprites.py:27-34: i0 layer the new sprites are appended to, i1 how many,
                                    i2,i3 ipool list of the LAYERS they must not overlap, i4 sampler table
                                    (as MOOG_Z_GENERATE), i5 dtype flags; MOOG_FL_DISJOINT / FAIL_GRACEFULLY,
                                    p0 max_recursion_depth; p2 > p1: the count is drawn per call from {p1 .. p2 - 1}
                                    with the uniform of rule-noise column p3.  Drawn on the device (Philox keyed by
                                    seed, env and a per-env serial) */
  MOOG_R_TREE,                   /* a user-defined rule class (functional_maze.py:18-67 `Booster`), its `step` traced along
                                    every path into a decision tree (node layout: MOOG_SC_TREE; kinds 3 = test
                                    `index < len(layer)`, 4 = run the stores of `expr` then go on; the leaf ends the
                                    rule): i0 ipool start, i1 nodes; the rule's own numeric attributes live in envf
                                    [i2, i2 + i3) and are set to dpool[i4 ...] when the rule is reset */
  MOOG_R_FIXATION,               /* fixation.py:45-54: i0 agent layer, i1 fixation layer (first sprite of each), i2 envf
                                    slot of meta_state[key], p0 threshold: += 1 while the two are closer, else 0 */
  MOOG_R_PHASESEQ_BEGIN,         /* task_phases.py:98-141 PhaseSequence: i0 envf slots (current phase index, its value
                                    when this pass began), i1 phases, i2 envf slot of meta_state[phase name key] or -1,
                                    i4 dpool index of the phases' name codes */
  MOOG_R_PHASE_BEGIN,            /* task_phases.py:18-95 Phase: guards the i1 ops that follow (a MOOG_R_COND_BEGIN on
                                    "first step" around the one-time rules, the continual rules, MOOG_R_PHASE_END);
                                    they run while the phase has not ended and -- i0 >= 0: envf slot pair of its
                                    PhaseSequence -- it is phase i2 of the sequence.  i3 envf slots (should_end,
                                    step_count, duration); the duration is p0, or (p2 > p1) drawn at reset from
                                    {p1 .. p2 - 1} with the uniform of rule-noise column i4 */
  MOOG_R_PHASE_END,              /* step_count += 1; ended when step_count >= duration or condition op i0 (-1: never)
                                    holds; then the sequence (i2 >= 0) moves on and names the next phase in envf[i3]
                                    (dpool[i4 + index], i5 phases; past the last one: the reference's IndexError).
                                    i1 envf slots of the phase */

  /* tasks: i[5] = envf slot of the countdown */
  MOOG_T_CONTACT_REWARD = 96, /* i0,i1 list0; i2,i3 list1; i4 cond expr; p0 reward p1 reset_steps; p2 > 0: the
                                 reward is the expression p2 - 1 of (sprite_0, sprite_1) instead of p0  contact_reward.py:70-102 */
  MOOG_T_RESET,               /* i0 condition op index; p0 steps_after p1 reward; i1 > 0: the reward is the value of
                                 condition op i1 - 1 (a reward_fn that reads the state)   reset.py:48-61  */
  MOOG_T_STAY_ALIVE,          /* p0 period p1 value                          stay_alive.py:22-32   */
  MOOG_T_TIMEOUT,             /* p0 timeout_steps                            composite_task.py:35  */

  /* action spaces: i0,i1 layer list; i2 offset in action vector; i5 envf slot */
  MOOG_A_JOYSTICK = 128,   /* p0 scaling p1 momentum      joystick.py:45-65    */
  MOOG_A_GRID,             /* p0 scaling p1 momentum      grid.py:52-70        */
  MOOG_A_SET_POSITION,     /* p0 inertia                  set_position.py:34-47 */

  /* device-side reset sampler (state_initialization/sprite_generators.py:26-105 for initializers
   * made of fixed sprites and generate_sprites groups): i0 first slot, i1 number of sprites,
   * i2,i3 ipool list of the slots the new sprites must not overlap (`without_overlapping`),
   * i4 ipool index of the sampler table (MOOG_Z_N_ATTRS entries of 3 ints: kind, dpool index, n),
   * flags MOOG_FL_DISJOINT / MOOG_FL_FAIL_GRACEFULLY, p0 max_recursion_depth; p2 > p1: the number of
 * sprites is drawn from {p1, ..., p2 - 1} per env and episode (`num_sprites=lambda:
 * np.random.randint(p1, p2)`), i1 being the largest count */
  MOOG_Z_GENERATE = 192,

  /* state conditions (value = double; used by MOOG_T_RESET / MOOG_R_COND_BEGIN) */
  MOOG_SC_ALL = 160,       /* i0,i1 layer list; i2 sprite expr: all(expr(s))   */
  MOOG_SC_ANY,             /* any(expr(s))                                     */
  MOOG_SC_COUNT,           /* sum(bool(expr(s)))                               */
  MOOG_SC_CONTACT_COUNT,   /* i0 layer0 i1 layer1: len(get_contact_indices)    contact_rules.py:38-51 */
  MOOG_SC_CONTACT_ANY_COUNT, /* i0,i1 list of sprites' layers; i2,i3 other list; i4 filter expr:
                                count of list-0 sprites passing the filter that overlap any list-1 sprite */
  MOOG_SC_CONST,           /* p0                                                */
  MOOG_SC_BINARY,          /* i0, i1 operand condition ops; i2 = MOOG_X_* binary opcode.  MOOG_X_AND /
                              MOOG_X_OR follow Python: the right operand is only evaluated when needed
                              (matters for the overlap calls a contact count makes) and the value is
                              that of the deciding operand */
  MOOG_SC_NOT,             /* i0 operand condition op: python `not`             */
  MOOG_SC_FIRST,           /* i0,i1 layer list; i2 sprite expr evaluated on the FIRST sprite of the list
                              (`state[layer][0]`); 0 when the list is empty      */
  MOOG_SC_BERNOULLI,       /* `np.random.binomial(1, p)` as a condition (first_person_predators_prey.py:181,189):
                              1 when the uniform in rule-noise column i0 is below p0 */
  MOOG_SC_TREE             /* a state-level callable that picks single sprites (`state['agent'][0]`), reads their
                              attributes / metadata, tests overlaps between them and branches
                              (bounce_box_contact_prediction.py:94-110), as a decision tree walked lazily from node
                              0 -- the overlap tests made are the ones Python would make, in its order.
                              i0 ipool start, i1 number of nodes of 8 ints:
                                kind (0 leaf: value = expr; 1 test expr != 0; 2 test overlaps(sprite 0, sprite 1)),
                                expr, layer and index of sprite 0, layer and index of sprite 1 (layer -1: unused),
                                next node if true, next node if false.
                              An index beyond the layer's count is the reference's IndexError: MOOG_ERR_BAD_INDEX */
};

/* op flags */
#define MOOG_FL_SYMMETRIC        1
#define MOOG_FL_UPDATE_ANGLE_VEL 2
#define MOOG_FL_APPLY_DISTANT    4
#define MOOG_FL_APPLY_NEARBY     8
#define MOOG_FL_HAS_ANCHOR       16
#define MOOG_FL_CONSTRAINED_LR   32
#define MOOG_FL_CONTROL_VELOCITY 64
#define MOOG_FL_SAMPLE_ONE       128
#define MOOG_FL_PREVENT_BACKTRACKING    256
#define MOOG_FL_ALLOW_WALL_BACKTRACKING 512
#define MOOG_FL_ONLY_TURN_AT_WALL       1024
#define MOOG_FL_DISJOINT                2048
#define MOOG_FL_FAIL_GRACEFULLY         4096

/* Sampler table of a MOOG_Z_GENERATE op: one entry per sprite factor in the order of the
 * MOOG_AT_* attribute ids, then the shape.  kind: constant (dpool[idx]); uniform: value =
 * float32(lo + (hi - lo) * u), lo = dpool[idx], hi = dpool[idx + 1] (distributions.py:71-90,
 * Continuous samples are float32); discrete: one of the n values dpool[idx ..] with equal
 * probability (for the shape entry the values are shape ids).
 * The table is followed by the extension program of the factors that are not drawn independently:
 * n_ext, then per component either [1, n_alt, dpool index of the cumulative probabilities, then per
 * alternative: n_leaves, (attr, kind, dpool index, n) ...] for a Mixture, or [2, keep_if_inside,
 * n_leaves, leaves ..., n_box, (attr, dpool index of lo hi) ...] for SetMinus (0) / Selection (1): the
 * base leaves are redrawn until the draw is outside / inside the box of Continuous ranges.
 * Shape record in dpool (one per distinct outline, sprite.py:329-424): [0] number of vertices nv,
 * [1] 1 if the shape is named 'circle', [2],[3] rotational inertia per unit mass about the centroid
 * (x, y parts), [4],[5] centroid of the raw outline (added to the position, sprite.py:389-406),
 * [6 ...] the nv centroid-centred vertices (x, y). */
#define MOOG_Z_N_ATTRS 14
#define MOOG_Z_SHAPE_ATTR 13
enum { MOOG_ZK_CONST = 0, MOOG_ZK_UNIFORM32 = 1, MOOG_ZK_DISCRETE = 2,
       MOOG_ZK_DISCRETE_P = 3 /* n candidates followed by their n cumulative probabilities (Discrete(probs=...)) */ };
#define MOOG_ERR_PORTAL_ODD      64u /* portal.py:49-52 ValueError: odd number of portals */
#define MOOG_ERR_BAD_INDEX      128u /* `state[layer][i]` with i >= len(state[layer]): the reference's IndexError */
#define MOOG_ERR_RESET_REJECTED  32u /* sprite_generators.py:92-98 RecursionError (no room for a sprite) */

/* Maze record in envf (maze_lib/maze.py:20-35, Maze.from_state :38-84, evaluated by the host when
 * a state is packed -- the wall sprites never move): [0] = maze_size N (<= MOOG_MAX_MAZE),
 * [1 + j] = row j as an integer whose bit i is maze[j, i] (1 = wall). */
#define MOOG_MAX_MAZE 32
#define MOOG_MAZE_WORDS (1 + MOOG_MAX_MAZE)

/* expression VM ------------------------------------------------------------ */
typedef struct {
  int32_t op;
  int32_t arg;
  double c;
} moog_ex; /* 16 bytes */

enum {
  MOOG_X_END = 0,
  MOOG_X_CONST,      /* push c                                              */
  MOOG_X_ATTR0,      /* push attribute `arg` of sprite 0 (see MOOG_AT_*)     */
  MOOG_X_ATTR1,      /* push attribute `arg` of sprite 1                     */
  MOOG_X_LT, MOOG_X_LE, MOOG_X_GT, MOOG_X_GE, MOOG_X_EQ, MOOG_X_NE,
  MOOG_X_AND, MOOG_X_OR, MOOG_X_NOT,
  MOOG_X_ADD, MOOG_X_SUB, MOOG_X_MUL, MOOG_X_DIV, MOOG_X_NEG, MOOG_X_ABS,
  MOOG_X_MOD,        /* python float modulo                                  */
  MOOG_X_STORE,      /* pop -> attribute `arg` of sprite 0 (modifier programs).  c: for `angle` the NumPy kind of
                        the value (sprite.py:531-540; 4 = whatever kind the angle has now); for `x_vel` / `y_vel` 3 = the components of a FRESH float64
                        array (`s.velocity = np.zeros(2)`, sprite.py:639-643): MOOG_SF_VEL32 and the alias id go */
  MOOG_X_STORE_POS,  /* pop y, pop x -> sprite 0 `.position = (x, y)`: one translation of the cached
                        outline (sprite.py:616-633) */
  MOOG_X_SELECT,     /* pop b, pop a, pop c -> (c != 0 ? a : b): an `if` / `else` of a config callable on a
                        per-sprite value, both sides traced (lambdas._explore) */
  MOOG_X_ENVF,       /* push envf[arg]: a state variable of a user-defined rule (MOOG_R_TREE) */
  MOOG_X_STORE_ENVF, /* pop -> envf[arg] */
  MOOG_X_RULE_NOISE, /* push this pass's uniform of rule-noise column arg: np.random.uniform / randint inside a traced
                        rule (match_to_sample.py:62-65) */
  MOOG_X_NORM2       /* pop y, pop x -> np.linalg.norm([x, y]) */
};

/* attribute ids for the expression VM (Sprite.FACTOR_NAMES, sprite.py:237-253) */
enum {
  MOOG_AT_X = 0, MOOG_AT_Y, MOOG_AT_X_VEL, MOOG_AT_Y_VEL, MOOG_AT_ANGLE,
  MOOG_AT_ANGLE_VEL, MOOG_AT_MASS, MOOG_AT_SCALE, MOOG_AT_ASPECT_RATIO,
  MOOG_AT_C0, MOOG_AT_C1, MOOG_AT_C2, MOOG_AT_OPACITY,
  MOOG_AT_META0 = 16 /* + k: column k of the sprite's numeric metadata (MOOG_H_META_OFF) */
};
#define MOOG_MAX_META 8

/* Sprite observation (RawState, raw_state.py:17-19), written by moog_observe_sprites:
 * float32 out[N][S][MOOG_OBS_COLS], slots in record order -- layers in state order, the sprites of a
 * layer in list order (z-order); layer l owns slots [layer_off[l], layer_off[l+1]) and its first
 * cnt[n][l] are live.  Columns 0-13 follow Sprite.FACTOR_NAMES (sprite.py:237-241) without metadata;
 * every value is the record's double rounded to nearest float32 (NaN stays NaN, inf stays inf).  A slot
 * that holds no sprite reads 0 in every column but MOOG_OBS_LAYER, whatever the record keeps there. */
#define MOOG_OBS_X 0          /* dyn  MOOG_D_X      */
#define MOOG_OBS_Y 1          /* dyn  MOOG_D_Y      */
#define MOOG_OBS_SHAPE 2      /* meta MOOG_M_SHAPE: shape id (BatchedEnvironment.shape_names) */
#define MOOG_OBS_ANGLE 3      /* dyn  MOOG_D_ANG    */
#define MOOG_OBS_SCALE 4      /* stat MOOG_S_SCALE  */
#define MOOG_OBS_ASPECT 5     /* stat MOOG_S_ASPECT */
#define MOOG_OBS_C0 6         /* stat MOOG_S_C0     */
#define MOOG_OBS_C1 7         /* stat MOOG_S_C1     */
#define MOOG_OBS_C2 8         /* stat MOOG_S_C2     */
#define MOOG_OBS_OPACITY 9    /* stat MOOG_S_OPACITY */
#define MOOG_OBS_X_VEL 10     /* dyn  MOOG_D_VX     */
#define MOOG_OBS_Y_VEL 11     /* dyn  MOOG_D_VY     */
#define MOOG_OBS_ANGLE_VEL 12 /* dyn  MOOG_D_ANGVEL */
#define MOOG_OBS_MASS 13      /* stat MOOG_S_MASS (inf stays inf) */
#define MOOG_OBS_LAYER 14     /* layer index of the slot, live or not */
#define MOOG_OBS_ALIVE 15     /* 1 for a live slot, 0 otherwise */
#define MOOG_OBS_COLS 16

/* step_type values written by the kernels (dm_env.StepType) */
enum { MOOG_STEP_FIRST = 0, MOOG_STEP_MID = 1, MOOG_STEP_LAST = 2 };

#ifdef __cplusplus
}
#endif
#endif /* MOOG_B200_PROGRAM_H_ */
