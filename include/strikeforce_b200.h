/*
 * strikeforce_b200.h -- C ABI of the B200-native batched StrikeForce simulator.
 *
 * The drop-in boundary for the reference's hot path (SURVEY.md section 8b).  The reference
 * has no FFI: bots plug in at compile time through `selected_agent.hpp` /
 * `selected_custom.hpp` (reference StrikeForce-client/selected_agent.hpp:25,
 * selected_custom.hpp:25, README.md:288-300) and the engine is the global
 * `gameplay g` (gameplay.hpp:437-1739).  Each entry point below names the reference
 * interface it replaces.  Plain pointers and sizes only; no C++ or torch types.
 *
 * Threading: a handle is bound to the CUDA device that was current in sf_create and is
 * not thread-safe; distinct handles (one per GPU) are independent.  All device work is
 * enqueued on the caller's stream (a cudaStream_t passed as void*, NULL = default stream).
 * Every call returns 0 on success, <0 on error (sf_last_error gives the text).
 * There is no CPU fallback: every compute entry point fails with SF_ERR_NO_DEVICE when
 * no CUDA device is usable.
 */
#ifndef STRIKEFORCE_B200_H
#define STRIKEFORCE_B200_H

#include <stdint.h>

#include "sf_canon.h"   /* status codes, game modes, canonical record */

#ifdef __cplusplus
extern "C" {
#endif

#define SF_ABI_VERSION 3

/* arena geometry: compile-time constants, as in the reference (gameplay.hpp:37: F = 3, N = 30, M = 100).
   A library for a larger map is the same source built with -DSF_ROWS= -DSF_COLS= (csrc/build.sh with
   SF_GEOMETRY=40x128 builds libstrikeforce_b200_40x128.so); rows x columns, rounded up to tiles of 4 x 8, must
   keep a cell id within 14 bits: 3 * ceil(rows / 4) * ceil(cols / 8) * 32 <= 16,384.  sf_config.map_cells /
   map_portal are [SF_CELLS] of the library they are handed to. */
#define SF_FLOORS 3
#ifndef SF_ROWS
#define SF_ROWS   30
#endif
#ifndef SF_COLS
#define SF_COLS   100
#endif
#define SF_CELLS  (SF_FLOORS * SF_ROWS * SF_COLS)

#define SF_OBS_CH   32                                   /* bots/bot-0.5/Custom.hpp:29-135 */
#define SF_OBS_WIN  31                                   /* bots/bot-0.5/Custom.hpp:142    */
#define SF_OBS_LEN  (SF_OBS_CH * SF_OBS_WIN * SF_OBS_WIN) /* 30,752 fp32                    */

#define SF_SHEET_LEN 32  /* character sheet without the name, Character.hpp:669-689:
                            3 defaults, 3 levels, money, 4 rates | 4 consumable counts |
                            4 x (throwable level, count) | 8 weapon levels | backpack level */

enum {
    SF_OK = 0,
    SF_ERR_ARG = -1,
    SF_ERR_NO_DEVICE = -2,   /* no CUDA device / driver: the product has no CPU path */
    SF_ERR_CUDA = -3,
    SF_ERR_UNSUPPORTED = -4,
    SF_ERR_NOMEM = -5
};

/* Items/cons*.txt: "name price vol lvl stamina | Hp effect" (Item.hpp:70-75) */
typedef struct sf_consumable { int32_t stamina, hp, effect; } sf_consumable;
/* Items/throw*.txt, Items/w*.txt: "... stamina | damage effect range" (Item.hpp:113-118,149-154) */
typedef struct sf_weapon { int32_t stamina, damage, effect, range; } sf_weapon;

/*
 * Everything `gameplay::setup()` + `load_data()` read from disk or from the menus
 * (gameplay.hpp:1231-1277, 1741-1925; Item.hpp:179-188; Character.hpp:650-709),
 * as plain arrays.  Replaces: map/floorK.txt, Items/\*.txt, character/\*.txt, the account sheet,
 * and the interactive mode / level prompts of gameplay::open() (gameplay.hpp:1507-1678).
 */
typedef struct sf_config {
    int32_t abi_version;             /* SF_ABI_VERSION */
    int32_t n_envs;                  /* arenas held by this handle */
    int64_t env_id_base;             /* global id of local arena 0 (multi-GPU sharding, SURVEY 8e) */
    int32_t mode;                    /* SF_MODE_SOLO / TIMER / SQUAD / ROYALE */
    int32_t level_min, level_max;    /* arena e plays level level_min + e % (level_max-level_min+1) */
    int32_t squad_agents;            /* 1: the 9 squad NPCs are driven (USE_AGENT_IN_SQUAD_NPCS,
                                        gameplay.hpp:1886-1901); 0: they idle ('+'), macros.hpp:14 */
    int32_t auto_reset;              /* 1: a terminal arena is re-created in the same step call */
    int32_t max_steps;               /* >0: truncate episodes (new behaviour)                  */
    /* slot capacities (reference: 9000 each, gameplay.hpp:37); exceeding one is SF_OVERFLOW   */
    int32_t cap_humans, cap_zombies, cap_bullets, cap_chests, cap_built, cap_portals;
    /* static map: one char per cell ('#', '.', '^', 'v', 'O'), row-major [floor][row][col],
       and the destination exit index of each '^' / 'v' (-1 elsewhere); gameplay.hpp:1252-1274 */
    const uint8_t *map_cells;        /* [SF_CELLS] host pointer */
    const int16_t *map_portal;       /* [SF_CELLS] host pointer */
    sf_consumable consumables[4];
    sf_weapon throwables[4];
    sf_weapon weapons[8];            /* level 0 stats; each owned level applies upgrade(), Item.hpp:105-111 */
    int32_t player_sheet[SF_SHEET_LEN]; /* the account sheet (me.build), Character.hpp:650-709 */
    int32_t npc_sheet[SF_SHEET_LEN];    /* character/human_enemy.txt (gen_human), Character.hpp:662-669 */
    /* SF_MODE_ROYALE (the reference's online modes as its replay reader plays them,
       gameplay.hpp:1795-1859): humans 0 .. royale_players-1 are players, every one of them with
       a sheet and a command of their own each step (sf_step: actions[env][player], any
       symbol of the alphabet); player i belongs to team royale_teams[i] (1..7); arena slot 0 is
       `ind` unless royale_ind says otherwise, the player whose death or victory ends the match: it carries
       player_sheet (hum[ind] = me), every other player i the sheet royale_sheets[i] it announced (get_info / scan_file,
       gameplay.hpp:131-149, 1797-1806).  Each player gets way = rand()%4+1 and a rejection-sampled
       '.' cell; the level is 1 (gameplay.hpp:1641, 1659). */
    int32_t royale_players;          /* 2..SF_MAX_PLAYERS */
    int32_t royale_teams[SF_MAX_PLAYERS];
    int32_t royale_sheets[SF_MAX_PLAYERS][SF_SHEET_LEN]; /* row royale_ind is not read */
    /* which player of a Battle Royale arena is `ind`, the player whose copy of the match this is
       (0 .. royale_players-1; 0 elsewhere): kill and loot credits go to `ind` and its team
       (gameplay.hpp:591-592, 629-630), its corpse keeps its cell (:642-645), its death or its team's
       victory ends the match, sf_step_out reports its Hp / damage / effect.  Every client of an online
       match holds such a copy; a match server that keeps one arena per seat sets this per handle. */
    int32_t royale_ind;
} sf_config;

typedef struct sf_handle sf_handle;

/* per-arena result of one step, written on the device ("reward" = integer deltas,
   SURVEY 8d: the reference has no scalar reward) */
typedef struct sf_step_out {
    int32_t status;        /* SF_RUNNING or the terminal status reached by this step            */
    int32_t d_kills;       /* gameplay::kills delta, gameplay.hpp:591-592, 629-630              */
    int32_t d_teams_kills; /* gameplay::teams_kills delta                                       */
    int32_t d_loot;        /* gameplay::loot delta                                              */
    int32_t d_hp;          /* main player Hp delta                                              */
    int32_t d_damage;      /* main player dealt-damage delta (Human::damage)                    */
    int32_t d_effect;      /* main player dealt-effect delta (Human::effect)                    */
    int32_t episode_steps; /* env-steps played in the episode (before any auto-reset)           */
} sf_step_out;

/* fields of sf_get */
enum {
    SF_FIELD_STEP_OUT   = 1, /* sf_step_out[n_envs]                                              */
    SF_FIELD_STATE_HASH = 2, /* uint64[n_envs]: sf_canon.h hash of each arena (parity checks)    */
    SF_FIELD_COUNTERS   = 3, /* int32[n_envs][8]: frame kills teams_kills loot chest steps status hp */
    SF_FIELD_POPULATION = 4, /* int32[n_envs][6]: humans zombies bullets chests built portals    */
    SF_FIELD_STATS      = 5, /* int64[16] device-reduced episode statistics (see SF_STAT_*)      */
    SF_FIELD_AGENT_OUT  = 6, /* sf_agent_out[n_envs][agents_per_env], after sf_enable_agent_out   */
    SF_FIELD_REPLAY     = 7, /* sf_replay_state[n_envs], after sf_enable_replay                   */
    SF_FIELD_REPLAY_DEALT = 8 /* uint8[n_envs][agents_per_env]: symbols dealt by the last step    */
};

/* slots of SF_FIELD_STATS: sums over the handle's arenas since sf_create (NCCL all-reduce
   these across GPUs; nothing else crosses devices, SURVEY 8e) */
enum {
    SF_STAT_STEPS = 0, SF_STAT_EPISODES, SF_STAT_WINS, SF_STAT_DEATHS, SF_STAT_TIMEOUTS,
    SF_STAT_TRUNCATED, SF_STAT_OVERFLOWS, SF_STAT_UB_GUARDS, SF_STAT_KILLS, SF_STAT_TEAMS_KILLS,
    SF_STAT_LOOT, SF_STAT_RNG_DRAWS, SF_STAT_ALGO_BYTES, SF_STAT_RESERVED0, SF_STAT_RESERVED1,
    SF_STAT_RESERVED2, SF_STAT_COUNT
};

/* observation points (SURVEY 7.4#7) */
enum { SF_OBS_P1 = 1 /* loop top, get_my_action gameplay.hpp:956 */,
       SF_OBS_P2 = 2 /* inside human_action, get_command gameplay.hpp:933 */,
       /* OR-ed into the phase: the same values with the channel innermost, [n_envs][n_obs_agents][31][31][32]
          (what a convolution library calls NHWC / channels-last; the reference's tensor, Custom.hpp:139, is
          [32][31][31]).  The policy's first convolution then reads the buffer as it is instead of
          transposing 123,008 bytes per observation first. */
       SF_OBS_NHWC = 0x100,
       /* OR-ed into the phase, at most one of the two, with or without SF_OBS_NHWC: obs holds 2-byte
          values, IEEE fp16 or bfloat16, in the same layout and for the same rows.  Element i is the
          round-to-nearest-even conversion of element i of the fp32 buffer the same call without the flag
          writes (61,504 B per observation instead of 123,008; SF_STAT_RESERVED0 counts as for fp32).  Every
          observation value is 0 or in [0.15, 12), so fp16 holds them without overflow or subnormals and keeps more
          of them distinct; bfloat16 is what a bf16 network reads without a cast.  Both flags set is
          SF_ERR_ARG, as is either flag for a library that predates them: a caller can probe for them. */
       SF_OBS_F16 = 0x200,
       SF_OBS_BF16 = 0x400 };

/* Replaces: the process-wide `gameplay g` and its globals (gameplay.hpp:47-55, 1739). */
int sf_create(const sf_config *cfg, sf_handle **out);
int sf_destroy(sf_handle *h);

/* Replaces gameplay::setup() + load_data() (gameplay.hpp:1231-1277, 1741-1925) for the listed
   local arenas (env_ids == NULL: all n_envs).  tb / serial are the two seeds of
   Random::_srand (random.hpp:64-76); NULL selects the synthetic seeds of sf_synth.h.
   env_ids, tb, serial are HOST arrays of length n. */
int sf_reset(sf_handle *h, const int32_t *env_ids, int32_t n, const int64_t *tb, const int64_t *serial,
             void *stream);

/* One env-step for every arena = one iteration of the loop in gameplay::play()
   (gameplay.hpp:1443-1472).  actions: DEVICE pointer, uint8 [n_envs][agents_per_env],
   each a command symbol of valid_commands (gameplay.hpp:45) or '_' ; replaces command[]
   (gameplay.hpp:43) as filled by get_my_action / get_command (gameplay.hpp:929-963). */
int sf_step(sf_handle *h, const uint8_t *actions, void *stream);

/* The two halves of sf_step (always called in pairs: a second sf_step_a, or sf_step, before the
   sf_step_b that closes the first is SF_ERR_ARG), for callers that need the P2 observation point
   (get_command -> bot() inside human_action, gameplay.hpp:933): sf_step_a runs the spawns and
   half-tick A (gameplay.hpp:1444-1461), sf_observe(..., SF_OBS_P2, ...) then sees what the
   squad agents see, and sf_step_b applies the actions and runs half-tick B (:1462-1471).
   sf_step_a then sf_step_b leaves every arena, its sf_step_out and the statistics exactly as sf_step
   would.  An arena whose episode ends in half A (SF_OVERFLOW, SF_UB_GUARD) keeps its terminal status
   until sf_step_b, which reports it and, with auto_reset, resets the arena at its end; its P2
   observation is undefined, as is the state after any abort. */
int sf_step_a(sf_handle *h, void *stream);
int sf_step_b(sf_handle *h, const uint8_t *actions, void *stream);

/* The same step through HOST buffers (the call a CPU-side trainer makes): takes the actions from
   actions_host, steps, delivers sf_step_out[n_envs] to out_host and synchronises.
   Page-locked buffers (cudaHostAlloc / cudaHostRegister) are used in place: the kernel reads each
   arena's commands from actions_host when human_action needs them and stores each arena's result
   into out_host while the other arenas are still stepping.  Pageable buffers are copied (host->device
   before, device->host after the step). */
int sf_step_host(sf_handle *h, const uint8_t *actions_host, sf_step_out *out_host, void *stream);

/* Fill a device action buffer with the synthetic stream of sf_synth.h for global step t. */
int sf_synth_actions(sf_handle *h, uint8_t *actions, uint64_t t, const char *table, int32_t table_len,
                     void *stream);

/* Replaces gameplay::bot() up to the Agent::predict call (bots/bot-0.5/Custom.hpp:137-158):
   writes the fp32 [n_envs][n_obs_agents][32][31][31] observation of the driven humans into the
   DEVICE buffer obs ([..][31][31][32] with phase | SF_OBS_NHWC; fp16 or bfloat16 values with phase |
   SF_OBS_F16 or phase | SF_OBS_BF16).  obs must be 16-byte aligned.  agent_mask bit a selects human slot a
   (bit 0 = the player).  phase names the
   observation point the caller is at and must match the handle: SF_OBS_P2 between sf_step_a and
   sf_step_b, SF_OBS_P1 otherwise (SF_ERR_ARG if it does not). */
int sf_observe(sf_handle *h, void *obs, int32_t phase, uint32_t agent_mask, void *stream);

/* Final observations and partial resets without the host (DESIGN.md section 7b).  With auto_reset = 0 an arena
   whose episode ends keeps its terminal state until it is reset, so it can be observed; these three calls find,
   observe and reset such arenas on the device, in stream order, without a host synchronisation (a loop of
   step, list, observe and reset can be captured in a CUDA graph).

   auto_reset = 0 with sf_reset_finished right after every step (after sf_step_b for a split step) leaves every
   arena, its sf_step_out, the statistics and the records of sf_save byte for byte as auto_reset = 1 does,
   including arenas that ended in half A (SF_OVERFLOW, SF_UB_GUARD).  Between the step and the reset,
   sf_observe, sf_observe_list, sf_get, sf_export_env and sf_save see the terminal state; the terminal state of
   an abort is undefined, as always.  Finished means: the arena's state has a status other than SF_RUNNING, as
   the last column of SF_FIELD_COUNTERS shows (sf_step_out only says what the last step did).

   The ids of the finished arenas that have not been reset since, ascending, into the DEVICE buffer
   env_ids [n_envs]; their number into the DEVICE int32 *count (both 4-byte aligned).  Allowed anywhere, also
   between sf_step_a and sf_step_b. */
int sf_list_finished(sf_handle *h, int32_t *env_ids, int32_t *count, void *stream);

/* Reset, on the device, exactly the arenas sf_list_finished would list now, as auto_reset = 1 would have at the
   end of the step in which they ended: next episode of the arena's own synthetic seed chain (episode + 1), level
   from its global id, the pending stream installed.  sf_step_out and the SF_STAT_* statistics stay as they are
   (the step that ended the episode counted it).  SF_ERR_ARG between sf_step_a and sf_step_b; with
   auto_reset = 1 it finds nothing to do. */
int sf_reset_finished(sf_handle *h, void *stream);

/* sf_observe for a DEVICE list of arenas: row i of obs ([n_max][n_selected][32][31][31], or channel-innermost
   with SF_OBS_NHWC or-ed into phase) is the observation of arena env_ids[i] (DEVICE int32 [n_max]), for
   i < min(*count, n_max) (count: DEVICE int32, NULL = n_max rows).  Rows from that bound up to n_max are not
   written.  Duplicate ids are allowed; an id outside [0, n_envs) gives an all-zero row.  1 <= n_max <= n_envs;
   the phase rule, the output formats and the 16-byte alignment of obs are those of sf_observe. */
int sf_observe_list(sf_handle *h, void *obs, int32_t phase, uint32_t agent_mask, const int32_t *env_ids,
                    const int32_t *count, int32_t n_max, void *stream);

/* sf_step for a DEVICE list of arenas (DESIGN.md section 7d): advance some arenas and hold the rest, e.g. the K
   children of a clone in a search, or the arenas an asynchronous actor has actions for.  The list rules are those
   of sf_observe_list: entries i < min(*count, n_max) of env_ids (DEVICE int32 [n_max]; count: DEVICE int32, NULL =
   n_max; both 4-byte aligned) are live, 1 <= n_max <= n_envs, and row i of actions (DEVICE uint8
   [n_max][agents_per_env], the symbols of sf_step) is the command row of arena env_ids[i].
   - A listed arena ends the call byte for byte as sf_step with that row would leave it: its state, auto-reset at
     the end of the step and the pending random stream included, its sf_step_out row and its sf_save record.
   - Every word of an unlisted arena is untouched, its sf_step_out row too (it still describes the last step that
     arena took).  The SF_STAT_* statistics add up over the stepped arenas only.
   - An id outside [0, n_envs) is skipped.  An id listed more than once is stepped once, with the row of its lowest
     list index; its later entries are ignored.  A skipped or ignored entry writes nothing and counts nothing.
   - SF_ERR_ARG between sf_step_a and sf_step_b, for a NULL actions or env_ids, a misaligned env_ids or count, and
     n_max out of range.  The call neither opens nor closes a split step.
   Stream order, no host synchronisation: the call can be captured in a CUDA graph.  A caller probes for it by
   looking the symbol up (SF_ABI_VERSION stays 3). */
int sf_step_list(sf_handle *h, const uint8_t *actions, const int32_t *env_ids, const int32_t *count, int32_t n_max,
                 void *stream);

/* Action masks (DESIGN.md section 7f): which commands would change the arena if a driven human obeyed them
   now, so that a search can skip children that equal the idle one and a policy can leave out commands that do
   nothing.  The alphabet, in bit order, is valid_commands (gameplay.hpp:45) in the reference's order, then '_':
   bit j of a mask word stands for SF_COMMANDS[j].

   For an arena and an agent slot a (a column of the action row; slot a drives human slot a):
   - Controllable: the slot's symbol reaches obey.  The arena's status is SF_RUNNING, human a is live, and a is
     ind, or a Battle Royale player slot that is not a random NPC, or a squad agent (a < agents_per_env) that is
     not a random NPC (the branches of human_action).  A slot that is not controllable gets mask 0.
   - Delivered symbol d(s): what human_action hands to obey.  s itself for ind and Battle Royale players; for
     squad agents s if s is one of "+xzqeawsd", '+' otherwise.
   - The bit of '+' is set for every controllable slot, so such a mask is never empty.
   - The bit of '_' is set iff the slot is controllable and d('_') = '_'.
   - Every other bit s is set iff the slot is controllable and the arena after obey(a, d(s)) differs from the
     arena after obey(a, '+'), both from the arena as stored now.  "Differs" means the canonical record
     (sf_canon.h) or the status differs; the teleport and the chest claim at the end of obey are part of both
     sides, and an SF_OVERFLOW that the command would cause is a difference.  '3' is never set.
   The mask describes the state at the time of the call and enforces nothing: sf_step obeys every symbol as
   before.  Between sf_step_a and sf_step_b (P2) the state is exactly what obey starts from, except for the
   humans that act before slot a in the same human_action.  At P1 (the loop top) half A of the next step
   (spawns, zombies, bullets) still runs before obey.  The call is allowed at both points. */
#define SF_COMMANDS "+qe3uzxawsdfghjkl;'cvbnm,./[]_"
#define SF_N_COMMANDS 30

/* The masks of every arena (env_ids NULL: rows = n_envs, count must be NULL and n_max = n_envs) or of a DEVICE
   list of arenas with the list rules of sf_observe_list: entries i < min(*count, n_max) of env_ids (DEVICE int32
   [n_max]; count: DEVICE int32, NULL = n_max) are live, row i belongs to arena env_ids[i], duplicates are
   allowed, an id outside [0, n_envs) gives an all-zero row, rows from the count up to n_max are not written,
   1 <= n_max <= n_envs.  mask: DEVICE uint32 [rows][agents_per_env]; mask, env_ids and count 4-byte aligned.
   One kernel launch in stream order, no host synchronisation, no device memory of its own; it writes nothing
   in the handle (state, sf_step_out, statistics and records stay as they are).  SF_ERR_ARG for a NULL mask,
   misalignment, n_max out of range and a count without env_ids.  A caller probes for it by looking the symbol
   up (SF_ABI_VERSION stays 3). */
int sf_action_mask(sf_handle *h, uint32_t *mask, const int32_t *env_ids, const int32_t *count, int32_t n_max,
                   void *stream);

/* Per-agent step outputs (DESIGN.md section 7g): what the last step did to each human the caller drives, for a
   trainer with one row per driven human (the 16 players of a Battle Royale arena, ind and the squad agents) --
   sf_step_out describes ind alone.  Row (e, a), for arena e and agent slot a (0 <= a < agents_per_env; column a
   of the action row drives human slot a), describes the last step arena e took through sf_step, sf_step_a +
   sf_step_b, sf_step_host or sf_step_list (as a listed arena):
   - SF_AGENT_DRIVEN: slot a was controllable in the state the step started from -- the arena was SF_RUNNING,
     human a was live, and a is ind, or a Battle Royale player or a squad agent (a < agents_per_env) that is not a
     random NPC.  This is the rule of sf_action_mask: DRIVEN is exactly "the sf_action_mask word was not 0" just
     before the step.
   - SF_AGENT_DIED: DRIVEN, and human a was not live at the end of the step (every way the tick removes a human,
     '_' included), read before any auto-reset.
   - d_hp, d_damage, d_effect, d_kills: Hp, Human::damage, Human::effect and Human::kills of human slot a at the end
     of the step (before any auto-reset) minus at its start.  damage and effect are what the human dealt; kills
     counts the other-team humans and the zombies it killed (gameplay.hpp:574-634).
   - A slot that is not DRIVEN gets an all-zero row, e.g. every slot of an arena that had ended and waits for
     sf_reset_finished.  When row ind is DRIVEN, its d_hp, d_damage and d_effect equal the step's sf_step_out.
   - After an SF_OVERFLOW or SF_UB_GUARD step only SF_AGENT_DRIVEN is defined (the state is undefined as well).
   - Rows are those of the last step: sf_step_list leaves the rows of unlisted arenas alone, and sf_reset,
     sf_reset_finished, sf_load and sf_load_list do not touch rows.  They are not part of an arena record.
     Between sf_step_a and sf_step_b the rows are unspecified.
   The values are taken inside the step kernel: a slot freed by a death can hold a spawned NPC a step later, and
   auto-reset re-creates an arena before the step returns, so reading the state around a step cannot give them.
   With agent outputs on, the state, sf_step_out, the statistics and the records are byte for byte what they are
   without. */
typedef struct sf_agent_out {
    int32_t flags;    /* SF_AGENT_DRIVEN | SF_AGENT_DIED                      */
    int32_t d_hp;     /* Hp of human slot a: end of the step minus start       */
    int32_t d_damage; /* Human::damage delta (dealt), gameplay.hpp:574-634     */
    int32_t d_effect; /* Human::effect delta (dealt)                           */
    int32_t d_kills;  /* Human::kills delta (other-team humans and zombies)    */
} sf_agent_out;
enum { SF_AGENT_DRIVEN = 1, SF_AGENT_DIED = 2 };

/* Opt in to agent outputs, once per handle: allocates the handle's rows (n_envs * agents_per_env * 20 bytes of
   device memory, counted by sf_device_bytes), zeroed, and from then on every step call of the handle writes
   them.  A handle that never calls it runs the step kernels it always ran.  A second call does nothing;
   SF_ERR_ARG between sf_step_a and sf_step_b.  sf_get(SF_FIELD_AGENT_OUT) reads the rows (one kernel launch; it
   is SF_ERR_ARG before this call).  A caller probes for it by looking the symbol up (SF_ABI_VERSION stays 3). */
int sf_enable_agent_out(sf_handle *h);

/* Match logs (DESIGN.md section 7h): an opt-in per-arena tape of the command symbols the reference's logger writes
   to a .sf_sample file (gameplay.hpp:966-991), so that an episode played here can be written as a match log and
   replayed by the reference's client.  The tape of arena e holds the symbols of the episode e's last step played,
   in file order; each step of a running arena appends
   1. the symbol ind was given, actions[ind] as obey receives it, then
   2. in ascending slot order the symbol of every other human that is live when human_action gathers commands (the
      state after half-tick A) and is a Battle Royale player or a squad agent that is not a random NPC -- the rule
      of sf_action_mask on that state.  A squad agent's symbol is the delivered one: a symbol outside "+xzqeawsd"
      is logged as '+'.
   A tape restarts when a step begins with the arena's step count at 0; it then takes the episode's seeds (tb,
   serial: rebuilt from the term constants of the arena's stream; they seed the same stream, and equal the seeds
   of sf_reset below 10^18), level, episode counter and global id.  So sf_reset, auto-reset and sf_reset_finished
   do not touch tapes: after an auto-reset the tape still describes the finished episode until the arena's next
   step, and with auto_reset = 1 the arenas whose sf_step_out status is terminal are exported before the next step.
   sf_step_list appends for listed arenas only; the split step restarts in sf_step_a and appends in sf_step_b.
   sf_load and an accepted sf_load_list clear SF_LOG_COMPLETE on the arenas they overwrite.  Tapes are not part of
   arena records.  With logs on, the state, sf_step_out, agent outputs, statistics and records are byte for byte
   what they are without.
   An exported row is an sf_log_head followed by cap_symbols bytes of tape (the first n_symbols count), padded to
   a multiple of 16 bytes: sf_log_row_bytes. */
typedef struct sf_log_head {
    int32_t flags;     /* SF_LOG_*                                                              */
    int32_t status;    /* SF_RUNNING while the episode runs, then how it ended                  */
    int32_t level;     /* the episode's level (the offline format does not carry it)            */
    uint32_t episode;  /* the arena's episode counter                                           */
    int32_t steps;     /* steps since the restart, those past a full tape included              */
    int32_t n_symbols; /* symbols on the tape, at most cap_symbols                              */
    int64_t tb;        /* seeds of the episode's stream (Random::_srand), the log header        */
    int64_t serial;
    int64_t global_id; /* env_id_base + arena                                                   */
} sf_log_head;
enum {
    SF_LOG_COMPLETE = 1,     /* the tape holds every step since its restart, taken by this handle        */
    SF_LOG_TRUNCATED = 2,    /* the tape was full: later symbols were dropped (COMPLETE is cleared)      */
    SF_LOG_ABORTED = 4,      /* the episode ended in SF_OVERFLOW or SF_UB_GUARD                           */
    SF_LOG_UNREPLAYABLE = 8  /* a symbol the reference's reader (file >> char) skips: NUL or white space  */
};
#define SF_LOG_CAP_MAX (1 << 24) /* symbols per tape */

/* Opt in to match logs, once per handle: allocates n_envs rows of sf_log_row_bytes (counted by sf_device_bytes),
   zeroed (no tape is COMPLETE before its first restart), and from then on every step call of the handle records.
   SF_ERR_ARG between sf_step_a and sf_step_b, for cap_symbols outside [1, SF_LOG_CAP_MAX], and for a second call
   with another capacity; a second call with the same capacity does nothing.  A caller probes for it by looking the
   symbol up (SF_ABI_VERSION stays 3). */
int sf_enable_log(sf_handle *h, int32_t cap_symbols);

/* bytes of one exported row: sizeof(sf_log_head) + cap_symbols rounded up to 16; 0 before sf_enable_log */
int32_t sf_log_row_bytes(const sf_handle *h);

/* Export tapes into the DEVICE buffer rows (16-byte aligned), one launch, no host synchronisation.  env_ids ==
   NULL: row i is the tape of arena i, for every arena (n_max must be n_envs, count NULL).  Otherwise the list
   rules of sf_action_mask: row i < min(*count, n_max) (count read on the device; NULL = n_max) is the tape of
   arena env_ids[i], duplicates allowed, an id outside [0, n_envs) gives an all-zero row, rows beyond the count
   are not written.  Allowed at P1 and between sf_step_a and sf_step_b (the tape as it stands).  SF_ERR_ARG
   before sf_enable_log, for NULL rows, misalignment, n_max out of range and a count without env_ids. */
int sf_log_list(sf_handle *h, void *rows, const int32_t *env_ids, const int32_t *count, int32_t n_max, void *stream);

/* Replay (DESIGN.md section 7i): command tapes loaded into arenas and dealt by the step, the reading half of the
   match logs above.  A handle opts in once with sf_enable_replay(h, cap_symbols); every arena then has a replay
   tape and a replay state.
   Loading: sf_replay_load takes rows in the layout sf_log_list exports (an sf_log_head, then the symbols, padded to
   16 bytes; sf_replay_row_bytes equals sf_log_row_bytes of a handle with the same capacity, so an exported row loads
   as it is).  It reads tb, serial, level, episode and n_symbols of the head and ignores the other fields.  Loading a
   row into arena e resets e exactly as sf_reset(e, tb, serial) would, but with the head's level instead of the one
   the global id gives and the head's episode as the episode counter; then it copies the tape and arms it (cursor 0,
   SF_REPLAY_ARMED, steps 0, status SF_RUNNING).  A log this handle took, loaded back into the arena it came from,
   gives the same log again when logs are on.  An entry is refused for n_symbols outside [0, cap_symbols], tb < 0 or
   serial < 0, and a level outside [1, 64] (SF_MAX_LEVEL) or other than 1 on a Battle Royale handle.
   Dealing: every step call of a replay handle (sf_step, sf_step_a + sf_step_b, sf_step_host, and sf_step_list for
   the listed arenas) deals from armed tapes.  In human_action ind's symbol is the next tape symbol; then, in
   ascending slot order, each human the logger records (the humans of SF_CONTROLLABLE_RULE on the state after
   half-tick A other than ind: exactly those sf_log_list's tape appends for) takes the next tape symbol instead of
   its action-row entry.  A symbol dealt to a squad agent is delivered as an action-row symbol is: outside
   "+xzqeawsd" it becomes '+'.  Random NPCs and humans that are not recorded are not affected.  A step that needs a
   symbol past the end of the tape takes that symbol and the rest of its symbols from the action row, sets
   SF_REPLAY_EXHAUSTED and disarms the tape at the end of the step; later steps use the action rows.
   End: a step that leaves an armed arena in a terminal status sets SF_REPLAY_ENDED, records the status and disarms
   the tape, before any auto-reset; with symbols left over it also sets SF_REPLAY_SURPLUS (the replay left the
   recorded episode: another sheet, capacities, max_steps or level, or a tape that is not one episode).  With
   auto-reset the next episode follows the arena's own seed chain and the action rows.
   sf_reset, sf_load and an accepted sf_load_list disarm the tapes of the arenas they overwrite; sf_reset_finished
   does not touch the replay state.  Tapes and replay states are not part of arena records.
   Outputs: sf_get(SF_FIELD_REPLAY) gives sf_replay_state[n_envs]; sf_get(SF_FIELD_REPLAY_DEALT) gives uint8
   [n_envs][agents_per_env], entry a the symbol the arena's last step took from its tape for human slot a as it was
   delivered to obey, 0 for a slot that took none (every step of a replay handle writes the rows of the arenas it
   steps; unspecified between sf_step_a and sf_step_b).  Both are one launch and SF_ERR_ARG before the opt-in.
   On a replay handle with no tape armed the state, sf_step_out, agent outputs, logs, statistics and records are
   byte for byte those of a handle without replay; an armed tape makes the step ignore the action-row entry of
   every slot it deals to. */
typedef struct sf_replay_state {
    int32_t flags;     /* SF_REPLAY_*                                                       */
    int32_t cursor;    /* symbols dealt                                                     */
    int32_t n_symbols; /* symbols on the tape                                               */
    int32_t steps;     /* steps taken since the load                                        */
    int32_t status;    /* SF_RUNNING, or how the replayed episode ended                     */
} sf_replay_state;
enum {
    SF_REPLAY_ARMED = 1,     /* the next step deals from the tape                                 */
    SF_REPLAY_EXHAUSTED = 2, /* a step needed a symbol past the end of the tape                   */
    SF_REPLAY_ENDED = 4,     /* the replayed episode ended (status holds how)                     */
    SF_REPLAY_SURPLUS = 8    /* it ended with symbols left over                                   */
};

/* Opt in to replay, once per handle: allocates zeroed tapes and states (counted by sf_device_bytes).  SF_ERR_ARG
   between sf_step_a and sf_step_b, for cap_symbols outside [1, SF_LOG_CAP_MAX], and for a second call with another
   capacity; a second call with the same capacity does nothing.  Probed for by symbol (SF_ABI_VERSION stays 3). */
int sf_enable_replay(sf_handle *h, int32_t cap_symbols);

/* bytes of one load row (equal to sf_log_row_bytes for the same capacity); 0 before sf_enable_replay */
int32_t sf_replay_row_bytes(const sf_handle *h);

/* Load the DEVICE rows (16-byte aligned, sf_replay_row_bytes each) into arenas, in stream order with no host
   synchronisation (capturable in a CUDA graph), with the list rules and the all-or-nothing refusal of
   sf_load_list: row i < min(*count, n_max) (count NULL: n_max) goes to arena env_ids[i]; an id outside [0, n_envs)
   is skipped; a repeated id is loaded once, from its lowest live index; *status (device int32) becomes the number
   of refused owning entries, and nothing changes unless it is 0.  SF_ERR_ARG before sf_enable_replay, between
   sf_step_a and sf_step_b, for NULL or misaligned buffers and for n_max outside [1, n_envs]. */
int sf_replay_load(sf_handle *h, const void *rows, const int32_t *env_ids, const int32_t *count, int32_t n_max,
                   int32_t *status, void *stream);

/* Copy a per-arena field into a DEVICE buffer (sizes above). */
int sf_get(sf_handle *h, int32_t field, void *dev_out, void *stream);

/* Canonical record of one arena (sf_canon.h) into a HOST buffer; *n_inout = capacity in int32
   on entry, count on exit.  Synchronises. */
int sf_export_env(sf_handle *h, int32_t env, int32_t *host_buf, int64_t *n_inout);

/* Arena records: save arenas into a device buffer and put them back later, into the same handle or another
   one (search and branching, checkpoint and resume, rewind).  A record holds every per-arena word of the
   device state at the handle's full capacities -- pending random stream, both banks of the stream
   constants, dead slots, overlay hints and spill bits included -- behind a 64-byte header (magic, format
   version, record size, a fingerprint of the configuration, the global id env_id_base + env of the arena it
   was saved from).  The fingerprint covers what gives the state words their meaning (map geometry,
   capacities, mode, squad_agents, Battle Royale players and ind, templates and item tables, the static map);
   n_envs, env_id_base, auto_reset, max_steps and the level range are not part of it.  A record does not
   hold the handle's SF_STAT_* statistics: they stay sums over the steps this handle ran since sf_create.
   A checkpoint on disk is the records copied to the host as they are.

   Loading a record into an arena of the same global id (in any handle with the same fingerprint) restores
   it completely: it plays on exactly as its source would have, current episode, auto-resets and later
   episodes.  Loaded into another global id (a clone), the current episode goes on bit for bit, with the
   record's level and episode counter, but the seed chain stays with the slot: the pending stream is seeded
   again with the synthetic seeds (sf_synth.h) of the slot's global id for episode + 1, and from the next reset on the arena follows its own id's
   level and seeds, as if its previous episode had ended there (that first reset may finish the stream's
   warm-up in one go, as after sf_reset).  sf_observe, sf_get and sf_export_env of a loaded arena give what
   they gave for its source when it was saved, and sf_save of it gives back the loaded bytes (but for the
   header's global id after a clone).

   Host id arrays are checked on the host and staged in the handle; both calls synchronise before they
   return, and both are SF_ERR_ARG between sf_step_a and sf_step_b. */

/* bytes of one arena record of this handle (a multiple of 128; fixed for a given library build and
   configuration) */
int64_t sf_snapshot_bytes(const sf_handle *h);

/* Write the records of arenas env_ids[0..n) (HOST array; NULL = all n_envs in order, n ignored; at most n_envs
   entries) into the DEVICE buffer records, [n][sf_snapshot_bytes], 16-byte aligned.  Duplicate ids are
   allowed. */
int sf_save(sf_handle *h, const int32_t *env_ids, int32_t n, void *records, void *stream);

/* Overwrite arenas env_ids[i] (HOST array; NULL = all n_envs in order) with record rows[i] (HOST array; NULL =
   row i) of the DEVICE buffer records ([n_records][sf_snapshot_bytes], 16-byte aligned).  Destination ids must
   be distinct.  All or nothing: if any referenced record is not a record of a compatible handle (magic,
   version, size, fingerprint), no arena changes and the call returns SF_ERR_ARG. */
int sf_load(sf_handle *h, const int32_t *env_ids, int32_t n, const void *records, int32_t n_records,
            const int32_t *rows, void *stream);

/* sf_save / sf_load for a DEVICE list of arenas (DESIGN.md section 7e): the record calls of a search loop that
   runs on the device, e.g. clone a root into the K slots a policy picked and restore them afterwards, or a
   checkpoint of the arenas sf_list_finished just listed.  The list rules are those of sf_observe_list: entries
   i < min(*count, n_max) of env_ids (DEVICE int32 [n_max]; count: DEVICE int32, NULL = n_max; rows and status
   DEVICE int32 too; all 4-byte aligned) are live, 1 <= n_max <= n_envs; records is a DEVICE buffer
   [..][sf_snapshot_bytes], 16-byte aligned.  Stream order, no host synchronisation, no host-side state that
   changes between calls: both calls can be captured in a CUDA graph.  SF_ERR_ARG between sf_step_a and
   sf_step_b, for a NULL records or env_ids, misalignment and n_max out of range.  A caller probes for them by
   looking the symbols up (SF_ABI_VERSION stays 3).

   sf_save_list: row i of records becomes the record of arena env_ids[i] for every live i, byte for byte what
   sf_save writes for that id.  Duplicate ids are allowed; an id outside [0, n_envs) gives an all-zero row (magic
   0: no load accepts it).  Rows from min(*count, n_max) to n_max are not written.  One kernel launch.

   sf_load_list: arena env_ids[i] is overwritten with record row rows[i] (rows NULL: row i), as sf_load of that
   record would leave it (a record of another global id re-seeds the pending stream).  An id outside [0, n_envs)
   is skipped; an id listed more than once is loaded once, from its lowest live index; skipped and ignored
   entries are not checked and change nothing.  All or nothing, decided on the device: an owning entry is refused
   when its row is outside [0, n_records) or its record is not one of this configuration (magic, version, size,
   fingerprint), and if any is, no arena changes.  *status (DEVICE int32 [1]) is written by every call, the count
   of 0 included: the number of refused owning entries, so 0 means the listed arenas were loaded.  Every word of
   an unlisted arena is untouched; the SF_STAT_* statistics are not touched.  Also SF_ERR_ARG for a NULL status,
   n_records < 1 and rows == NULL with n_records < n_max.  A memset of *status and five kernel launches (claim,
   check, copy, re-seed, release), which share the claim words of sf_step_list: calls of one handle that use
   them (sf_step_list, sf_load_list) go to one stream. */
int sf_save_list(sf_handle *h, void *records, const int32_t *env_ids, const int32_t *count, int32_t n_max,
                 void *stream);
int sf_load_list(sf_handle *h, const void *records, int32_t n_records, const int32_t *rows,
                 const int32_t *env_ids, const int32_t *count, int32_t n_max, int32_t *status, void *stream);

/* Replaces Random::_srand + Random::_rand (random.hpp:54-76) for a batch of independent
   streams: seeds stream i with (tb[i], serial[i]) and writes n_draws outputs per stream into
   the HOST buffer out_host[draw * n_streams + i].  Known-answer tests use it. */
int sf_rng_stream(sf_handle *h, const int64_t *tb, const int64_t *serial, int32_t n_streams, int32_t n_draws,
                  int32_t *out_host);

int32_t sf_agents_per_env(const sf_handle *h);
int32_t sf_num_envs(const sf_handle *h);
/* kernels launched by this handle since creation (bench.py's gpu_launches claim) */
int64_t sf_launch_count(const sf_handle *h);
/* bytes of HBM held by the handle */
int64_t sf_device_bytes(const sf_handle *h);

const char *sf_last_error(const sf_handle *h);   /* h == NULL: last sf_create error */
int32_t sf_abi_version(void);

#ifdef __cplusplus
}
#endif

#endif /* STRIKEFORCE_B200_H */
