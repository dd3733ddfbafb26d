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
    SF_FIELD_STATS      = 5  /* int64[16] device-reduced episode statistics (see SF_STAT_*)      */
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
       SF_OBS_NHWC = 0x100 };

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
   DEVICE buffer obs ([..][31][31][32] with phase | SF_OBS_NHWC).  agent_mask bit a selects human slot a
   (bit 0 = the player).  phase names the
   observation point the caller is at and must match the handle: SF_OBS_P2 between sf_step_a and
   sf_step_b, SF_OBS_P1 otherwise (SF_ERR_ARG if it does not). */
int sf_observe(sf_handle *h, float *obs, int32_t phase, uint32_t agent_mask, void *stream);

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
   the phase rule and the 16-byte alignment of obs are those of sf_observe. */
int sf_observe_list(sf_handle *h, float *obs, int32_t phase, uint32_t agent_mask, const int32_t *env_ids,
                    const int32_t *count, int32_t n_max, void *stream);

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
