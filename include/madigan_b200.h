/*
 * madigan_b200.h -- C ABI of the B200-native batched Madigan environment.
 *
 * This is the drop-in boundary for Madigan's Env.step hot path.  The reference
 * exposes that path as the pybind11 module `env` (reference:
 * madigan/environments/cpp/env.cpp:843-1005 binds Env; Env::step is
 * madigan/environments/cpp/Env.h:189-256, Env::reset is Env.h:181-187).  Here the
 * same operations act on N independent environments whose state lives in HBM as
 * structure-of-arrays tensors owned by the caller (torch); the library is a set
 * of stateless launchers: it allocates nothing and keeps nothing between calls
 * except a thread-local error string.
 *
 * Conventions
 *   - every pointer in MdgState / MdgStepIO / MdgDerived is a DEVICE pointer;
 *   - per-env vectors are stored asset-major: field[a * n_envs + e]
 *     ("[nA][N]"), so that one warp touches one contiguous 256-byte run;
 *   - every launcher enqueues on `stream` (a cudaStream_t passed as void*) and
 *     returns without synchronising; return value 0 = ok, <0 = MDG_E_*.
 *   - arithmetic is IEEE fp64 without FMA contraction, sums run left to right
 *     over the asset index (the conventions of oracle/mdg_oracle.c).
 */
#ifndef MADIGAN_B200_H_
#define MADIGAN_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MDG_ABI_VERSION 16
#define MDG_MAX_ASSETS 16
#define MDG_GEN_NPARAM 10
#define MDG_BROKER_NPARAM 7 /* broker settings per set (MdgBrokerSlot): rows of a broker table */
#define MDG_MAX_NSTEP 64
#define MDG_MAX_SINE_COMPONENTS 16 /* 3 random bools per component share one 53-bit uniform */
#define MDG_MAX_SINE_TRENDS 4

/* error codes (reference: C++ exceptions translated by pybind11, DataTypes.h:36-46) */
#define MDG_OK 0
#define MDG_E_INVALID (-1)     /* bad argument / config  -> ValueError / RuntimeError */
#define MDG_E_UNSUPPORTED (-2) /* shape outside what the kernels were built for     */
#define MDG_E_CUDA (-3)        /* CUDA runtime error, text in mdg_last_error()      */

/* RiskInfo, declaration order of DataTypes.h:70-75 */
#define MDG_RISK_GREEN 0
#define MDG_RISK_INSUFF_MARGIN 1
#define MDG_RISK_MARGIN_CALL 2
#define MDG_RISK_BLOWN_OUT 3

/* synthetic generators (reference: DataSource.cpp makeDataSource :9-108) */
enum MdgGenType {
  MDG_GEN_SYNTH = 0,       /* DataSource.cpp:535-543  */
  MDG_GEN_OU = 1,          /* DataSource.cpp:1173-1180 */
  MDG_GEN_OUPAIR = 2,      /* DataSource.cpp:1232-1246 */
  MDG_GEN_SIMPLETREND = 3, /* DataSource.cpp:1324-1359 */
  MDG_GEN_TRENDOU = 4,     /* DataSource.cpp:1457-1502 */
  MDG_GEN_TRENDYOU = 5,    /* DataSource.cpp:1602-1657 */
  MDG_GEN_SAWTOOTH = 6,    /* DataSource.cpp:558-567  */
  MDG_GEN_TRIANGLE = 7,    /* DataSource.cpp:569-578  */
  MDG_GEN_GAUSSIAN = 8,    /* DataSource.cpp:1108-1114 */
  MDG_GEN_SINEADDER = 9,   /* DataSource.cpp:663-673  */
  MDG_GEN_SINEDYNAMIC = 10,     /* DataSource.cpp:802-841 + WaveTableOsc.h */
  MDG_GEN_SINEDYNAMICTREND = 11 /* DataSource.cpp:1002-1047 */
};

/* parameter slots p[] per generator type
 *  SYNTH/SAWTOOTH/TRIANGLE: 0 freq 1 mu 2 amp 3 phase(initial x) 4 dX 5 noise
 *  OU:          0 mean 1 theta 2 phi
 *  OUPAIR:      0 theta 1 phi 2 noise           (same on both assets of a pair)
 *  SIMPLETREND: 0 trendProb 1 minPeriod 2 maxPeriod 3 noise 4 start 5 dYMin 6 dYMax
 *  TRENDOU/TRENDYOU: 0 trendProb 1 minPeriod 2 maxPeriod 3 dYMin 4 dYMax 5 start
 *                    6 theta 7 phi 8 noiseTrend 9 emaAlpha(unused by the reference)
 *  GAUSSIAN:    0 mean 1 var(used as stddev)
 *  SINEADDER:   0 K (components) 1 offset into MdgParams.gen_ext 2 dX 3 noise
 *               gen_ext[off + 4c ..]: freq, mu, amp, phase of component c
 *  SINEDYNAMIC: 0 K 1 offset into gen_ext 2 sampleRate = (int)(1/dX) 3 noise
 *               gen_ext[off + 12c ..]: freq lo,hi,step; mu lo,hi,step; amp lo,hi,step; number of wave
 *               tables; offset of the component's table list; 0.  Table list entry (3 doubles): topFreq,
 *               len, offset of the len+1 samples (WaveTableOsc.h:126-157: sin(i 2 pi / len), last = first).
 *               The host builds the samples with libm's sin, so the oracle and the kernels interpolate
 *               the same doubles.
 *  SINEDYNAMICTREND: as SINEDYNAMIC, plus 4 T (trends) 5 offset of the trend list in gen_ext
 *               (4 doubles per trend: min length, max length, increment, probability)
 * generator-state rows (gstate) per asset, starting at gslot
 *  SYNTH/SAWTOOTH/TRIANGLE: x          OU/GAUSSIAN: none
 *  OUPAIR role 0: shared mean          OUPAIR role 1: none (uses partner's row)
 *  SIMPLETREND: dY, flags              TRENDOU: ouMean, dY, flags
 *  TRENDYOU: ouComponent, trendComponent, dY, flags
 *  SINEADDER: x of each component (K rows)
 *  SINEDYNAMIC: freq, mu, amp, phasor of each component (4K rows)
 *  SINEDYNAMICTREND: the 4K rows, trendComponent, one flags row per trend
 *  flags (int64 stored in the double row): bit0 trending, bit1 direction(+1),
 *  bits 32..63 remaining trend length.
 * noise slots: nslot = this asset's normal draw; nslot_aux = OUPair role 0 shared
 * random-walk draw (pair order rw,x0,x1 = DataSource.cpp:1233-1235); uslot = first
 * of 4 uniform slots (trigger, direction, length, dY) for the trend generators.
 * SINEADDER draws K normals (nslot + c).  SINEDYNAMIC(TREND) draws one normal and its random booleans
 * (randomBoolGenerator.h:8-14; 3 per component in the order mu, amp, freq, then one direction per trend)
 * from ONE uniform at uslot: boolean b is bit 52-b of floor(u 2^53).  SINEDYNAMICTREND then uses uslot+1+2j
 * (trend-start test) and uslot+2+2j (trend length) for trend j.  The uniform_real draws of the constructor
 * and of reset() (freq, mu, amp of every component, DataSource.cpp:771-773,783-787) come from Philox streams
 * 3 and 2 at the env's current tick, slot 64*asset + 3c + {0,1,2}.
 */
typedef struct MdgAssetGen {
  int32_t type;
  int32_t role;
  int32_t nslot;
  int32_t nslot_aux;
  int32_t uslot;
  int32_t gslot;
  int32_t partner;
  int32_t _pad;
  double p[MDG_GEN_NPARAM];
} MdgAssetGen;

/* per-batch constants (reference: Env.h:94-111 setters, Broker.cpp:78-85) */
typedef struct MdgParams {
  int32_t n_assets;
  int32_t n_gstate;   /* rows of generator state per env            */
  int32_t n_normals;  /* normal draws per env per tick (fixed slots) */
  int32_t n_uniforms; /* uniform draws per env per tick              */
  double init_cash;
  double required_margin;
  double maintenance_margin;
  double slippage_rel, slippage_abs;
  double tcost_rel, tcost_abs;
  MdgAssetGen gen[MDG_MAX_ASSETS];
  const double *gen_ext; /* device memory: parameter/wave tables of the SINE* generators, or NULL */
  int64_t n_gen_ext;     /* doubles in gen_ext */
} MdgParams;

/* reward shaping (reference: utils/buffers/nstep_buffer.py:23-312,378-408 and the
 * agent reward of modelling/algorithm/offpolicy_q.py:140-164) */
enum MdgShaper {
  MDG_SHAPER_OFF = 0, /* agent/shaped rewards not computed              */
  MDG_SHAPER_SUM = 1, /* sum_default                                    */
  MDG_SHAPER_DSR = 2,
  MDG_SHAPER_DDR = 3,
  MDG_SHAPER_COSINE = 4, /* cosine_port_shaper == the paper's PPC       */
  MDG_SHAPER_SHARPE = 5,
  MDG_SHAPER_SORTINO_A = 6,
  MDG_SHAPER_SORTINO_B = 7
};
typedef struct MdgReward {
  int32_t shaper;
  int32_t reduce_rewards; /* agent_config.reduce_rewards: sum per-asset rewards */
  int32_t nstep;          /* agent_config.nstep_return, 1..MDG_MAX_NSTEP        */
  int32_t _pad;
  double discount;
  double adaptation_rate;
  double cosine_temp;
  double sortino_exp;
  double desired_portfolio[MDG_MAX_ASSETS + 1];
  double discounts[MDG_MAX_NSTEP]; /* math.pow(discount, i), filled by the host exactly as nstep_buffer.py:330 */
} MdgReward;

/* persistent per-env state, all [rows][N].
 * Layout hint: when price, ledger, mean_entry and borrowed are equally spaced (views of one [4][nA][N] slab, 16-byte
 * aligned, N a multiple of 128) the all-OU-pairs step kernel fetches a pair's eight state rows with ONE 3-D TMA tensor
 * copy and the caller's units with a 2-D one; any other placement is accepted and read with plain loads. */
typedef struct MdgState {
  double *price;      /* [nA][N] currentPrices (== currentData for synthetic sources) */
  double *ledger;     /* [nA][N] Portfolio::ledger_          */
  double *mean_entry; /* [nA][N] Portfolio::meanEntryPrices_ */
  double *borrowed;   /* [nA][N] Portfolio::borrowedMargin_  */
  double *cash;       /* [N]     Portfolio::cash_            */
  double *gstate;     /* [n_gstate][N] generator state       */
  int64_t *timestamp; /* [N] generator tick counter          */
  double *shaper_A;   /* [ra][N] DSR/DDR moving first moment  (nullable)   */
  double *shaper_B;   /* [ra][N] DSR/DDR moving second moment (nullable)   */
  double *nstep_ring; /* [nstep][ra][N] raw rewards waiting in the n-step buffer (nullable when nstep==1) */
  int32_t *nstep_len; /* [N] entries currently in the n-step buffer          (nullable when nstep==1) */
  int64_t *reset_ts;  /* [N] timestamp at the end of the env's last reset: window rows older than that come
                         from MdgStepIO.pre_price (portfolio rows: flat [1,0,...,0]); the timestamp of a
                         window row is timestamp - age (every ring/prefix row is exactly one generator tick) */
  double *folds;      /* [5][N] cache of the portfolio's left-to-right folds at the current prices:
                         assetValue, meanEntry.ledger, sum borrowedMargin, short entry value, and a
                         magnitude bound.  Written by mdg_step / mdg_reset / mdg_init_state; call
                         mdg_refresh_folds after modifying price/ledger/mean_entry/borrowed/cash from outside. */
} MdgState;

/* inputs and outputs of one step / reset */
typedef struct MdgStepIO {
  const double *units;    /* step input: (N,nA) row-major transaction units; single-asset mode: (N,) */
  const double *normals;  /* nullable. validation mode: [ticks][n_normals][N] standard normals  */
  const double *uniforms; /* nullable. validation mode: [ticks][n_uniforms][N] uniforms in [0,1) */
  double *obs_price;      /* ring [k][nA][N]   State.price rows      */
  double *obs_port;       /* ring [k][nA+1][N] State.portfolio rows (ledgerNormedFull) */
  double *pre_price;      /* [N][k][nA] price rows of the last reset's history fill, env-major: a reset
                             rewrites an env's whole window, and k*nA scattered 8-byte writes into the
                             env-minor ring cost 8x their size in HBM traffic (sector read-modify-write),
                             so those rows live here, contiguous per env; row k-1 is the newest.  The ring
                             keeps only rows written by steps (and the newest row, = current state). */
  double *reward;         /* [N]  Env::step reward (log equity return, clamped) */
  uint8_t *done;          /* [N]                                       */
  double *trans_price;    /* [nA][N] BrokerResponse.transactionPrice   */
  double *trans_units;    /* [nA][N] BrokerResponse.transactionUnits   */
  double *trans_cost;     /* [nA][N] BrokerResponse.transactionCost    */
  uint8_t *risk;          /* [nA][N] BrokerResponse.riskInfo           */
  uint8_t *margin_call;   /* [N]     BrokerResponse.marginCall         */
  double *agent_reward;   /* [ra][N] offpolicy_q.py:153-164 (nullable when shaper off) */
  double *shaped_reward;  /* [nstep][ra][N] rewards popped from the n-step buffer this step (row j = j-th pop) */
  int32_t *n_popped;      /* [N] how many rows of shaped_reward are valid this step      */
  const int8_t *actions;  /* nullable, MDG_MODE_MULTI only: (N,nA) row-major discrete actions in [0, action_atoms).
                             When given, `units` is ignored and the transaction units are derived in the kernel as
                             DQN.action_to_transaction does (modelling/algorithm/dqn.py:160-179), from the portfolio
                             as it stands before the first transaction:
                               units_i = (a_i - action_atoms/2) * ((unit_size * availableMargin) / price_i),
                               a_i == 0 closes the position (units_i = -ledger_i, or 0 when flat). */
  const float *weights;   /* nullable, MDG_MODE_MULTI only: (N,nA+1) row-major fp32 target portfolio weights (cash first),
                             what a DDPG actor emits.  When given, `units` and `actions` are ignored and the units are
                             derived in the kernel as DDPG.action_to_transaction does (modelling/algorithm/ddpg.py:182-207)
                             from the portfolio as it stands before the first transaction:
                               desired = w / sum(w) (fp32; w itself when the sum is 0),
                               units_i = ((desired_{i+1} - ledgerNormedFull_{i+1}) * equity) / price_i. */
} MdgStepIO;

#define MDG_MODE_HOLD 0   /* Env::step()            Env.h:189-204 */
#define MDG_MODE_MULTI 1  /* Env::step(units)       Env.h:206-230 */
#define MDG_MODE_SINGLE 2 /* Env::step(idx, units)  Env.h:232-256 */

typedef struct MdgLaunch {
  int64_t n_envs;      /* envs in this slab                                   */
  int64_t env_offset;  /* global id of env 0 (Philox counter), for sharding   */
  uint64_t seed;       /* Philox key                                          */
  int32_t window;      /* k, rows in the observation ring                     */
  int32_t head;        /* ring slot that receives the newest row              */
  int32_t mode;        /* MDG_MODE_*                                          */
  int32_t asset_idx;   /* MDG_MODE_SINGLE only                                */
  int32_t nstep_pos;   /* physical n-step ring slot of the entry added now    */
  int32_t action_atoms; /* MdgStepIO.actions only: number of discrete actions per asset (dqn.py:166) */
  void *stream;        /* cudaStream_t                                        */
  double unit_size;    /* MdgStepIO.actions only: fraction of availableMargin per action unit (dqn.py:164) */
  int32_t flags;       /* MDG_FLAG_*                                          */
  int32_t _pad;
} MdgLaunch;
/* validation: every risk gate of mdg_step takes the exact left-to-right fold path (the cold path that otherwise
 * only decides knife-edge cases); ledgers must be identical with and without it */
#define MDG_FLAG_FORCE_EXACT_GATE 1
/* validation: refills (mdg_reset_ws, mdg_step_autoreset) take the generic kernel, also for parameter sets that have a
 * specialised one (all OU pairs); the results must be identical */
#define MDG_FLAG_GENERIC_FILL 2

/* derived accounting, Portfolio.cpp:140-235,243-252; any pointer may be NULL */
typedef struct MdgDerived {
  double *equity, *asset_value, *pnl, *balance, *available_margin, *used_margin;
  double *borrowed_margin, *borrowed_asset_value; /* [N] each */
  uint8_t *risk;                                   /* [N] Portfolio::checkRisk() */
  double *position_values, *pnl_positions, *ledger_normed, *ledger_abs_normed; /* [nA][N]   */
  double *ledger_normed_full, *ledger_abs_normed_full, *position_values_full,
      *ledger_full;                                                             /* [nA+1][N] */
} MdgDerived;

/* window normalisers, utils/preprocessor.py:53-107 */
enum MdgNorm {
  MDG_NORM_NONE = 0,
  MDG_NORM_LOOKBACK = 1,
  MDG_NORM_LOOKBACK_LOG = 2,
  MDG_NORM_LOG = 3,
  MDG_NORM_STANDARD = 4,
  MDG_NORM_LOG_STANDARD = 5,
  MDG_NORM_EXPANDING = 6
};
#define MDG_DTYPE_F64 0
#define MDG_DTYPE_F32 1
#define MDG_LAYOUT_NKF 0 /* (N,k,F) as StackerDiscrete.current_data, preprocessor.py:183-189 */
#define MDG_LAYOUT_NFK 1 /* (N,F,k) channels-first, what modelling/net/common.py:239-240 transposes to */

/* per-slab episode statistics, see mdg_episode_stats */
#define MDG_STATS_NSCALAR 8 /* count, sum_equity, sum_sq_equity, min_equity, max_equity, sum_reward, sum_cost, n_done */

int mdg_abi_version(void);
/* sizeof of the ABI structs as compiled: 0 MdgAssetGen 1 MdgParams 2 MdgReward 3 MdgState 4 MdgStepIO
 * 5 MdgLaunch 6 MdgDerived 7 MdgWindow 8 MdgReplay 9 MdgReplayBatch 10 MdgRewardNorm 11 MdgTearsheet
 * 12 MdgPrioritized 13 MdgReplayRows 14 MdgParamSets 15 MdgSetDraw 16 MdgEpisodeResults; -1 for an unknown index
 * (lets a binding verify its struct mirror) */
int mdg_sizeof(int which);
const char *mdg_last_error(void);

/* Env::step for every env of the slab: transact -> generator tick -> reward/done ->
 * newest observation row -> agent reward -> n-step shaped reward.
 * Replaces Env.h:189-256 + Broker.cpp:124-178 + Portfolio.cpp:243-323 +
 * DataSource.cpp getData family + offpolicy_q.py:140-164 + nstep_buffer.py:23-312. */
int mdg_step(const MdgParams *params, const MdgReward *reward, const MdgState *state,
             const MdgStepIO *io, const MdgLaunch *launch);

/* Env::reset (Env.h:181-187) for the envs with mask[e]!=0 (mask==NULL: all):
 * generator reset, fresh portfolio, one tick, and -- when fill_ticks>1 -- the
 * fill_ticks-1 no-action ticks of StackerDiscrete.initialize_history
 * (preprocessor.py:191-194); the rows end at ring slot launch->head.
 * clear_nstep!=0 also empties the n-step buffer (offpolicy_q.py:94). */
int mdg_reset(const MdgParams *params, const MdgState *state, const MdgStepIO *io,
              const MdgLaunch *launch, const uint8_t *mask, int fill_ticks, int clear_nstep);

/* Same operation with a caller-provided device workspace (at least mdg_reset_workspace_bytes): the
 * resetting envs are compacted into a list and ONE kernel refills them, a block per listed env (Philox +
 * Box-Muller of the whole history packed over the block into shared memory, then the serial recurrences of the
 * env's generator groups on neighbouring lanes) -- many times faster than mdg_reset when a few percent of the
 * envs reset every step.  When every asset belongs to an OU pair, there are at least 8 assets and the normals
 * come from Philox, the refill runs one lane per (env, pair) instead, with bit-identical results
 * (MDG_FLAG_GENERIC_FILL forces the generic kernel).  workspace == NULL falls back to mdg_reset.  The first 256 bytes of the workspace are a
 * header (list length, exit ticket) that must be ZERO before the first use; every call leaves it zero again. */
int mdg_reset_ws(const MdgParams *params, const MdgState *state, const MdgStepIO *io,
                 const MdgLaunch *launch, const uint8_t *mask, int fill_ticks, int clear_nstep,
                 void *workspace, int64_t workspace_bytes);
int64_t mdg_reset_workspace_bytes(const MdgParams *params, int64_t n_envs, int fill_ticks);

/* The agent loop's `step; if done: reset + initialize_history` (offpolicy_q.py:93-99,140-153) as ONE host call
 * and TWO launches: the step kernel appends the envs that finished to the workspace's list, the refill kernel
 * resets exactly those (its grid is sized without knowing the count; blocks past the end of the list exit at once).
 * `workspace` as for mdg_reset_ws (zeroed header before the first use), required. */
int mdg_step_autoreset(const MdgParams *params, const MdgReward *reward, const MdgState *state,
                       const MdgStepIO *io, const MdgLaunch *launch, int fill_ticks, int clear_nstep,
                       void *workspace, int64_t workspace_bytes);

/* Constructor state (Env.h:139-165 before the first tick): generator start values,
 * empty ledger, cash=init_cash, timestamp=0, shaper state zero. */
int mdg_init_state(const MdgParams *params, const MdgReward *reward, const MdgState *state,
                   const MdgLaunch *launch);

/* ---------------------------------------------------------------------------------------------------
 * Generator parameter sets: the envs of one slab tick different markets (a sweep over settings, or a distribution of
 * markets for robust training) with the same types, roles and slots; broker settings per set: the _sets_broker
 * launches below.
 *
 * A parameter set is one value for every p[j] slot (MDG_GEN_NPARAM) of every asset.  The table holds n_sets >= 1 of
 * them, set-minor: p[(i * MDG_GEN_NPARAM + j) * n_sets + s] is slot j of asset i in set s, so that a warp's reads
 * are coalesced when every env has its own set (n_sets == n_envs, set_of_env[e] == e) and stay on one 128-byte line
 * when n_sets <= 16.  Env e reads set s = set_of_env[e]; an index outside [0, n_sets) is clamped, as an unsigned
 * value, to n_sets - 1, so no index reads outside the table.
 * With sets, every read of params->gen[i].p[j] by the step, refill and constructor kernels reads the table entry of
 * the env's set instead.  Nothing else changes: types, roles, noise / uniform slots, gslot, broker settings, rewards
 * and the Philox draws (keyed on seed, global env id and tick only).  So env e of a launch with sets is bit for bit
 * env e of a launch without sets whose params->gen[i].p are those of set s.  OUPair reads as without sets: role 0
 * supplies p[2] (the shared mean's noise), each asset its own p[0] (theta) and p[1] (phi).
 * The SINE* types are not accepted (their p slots are component counts and offsets into gen_ext):
 * MDG_E_UNSUPPORTED.  params->gen[i].p must still be filled (the base set: the host-side checks read it).
 * The table and the assignment are read by each launch on its stream: a change made between launches takes effect at
 * the next launch, and an episode in progress continues under the new values. */
typedef struct MdgParamSets {
  const double *p;           /* device: [nA][MDG_GEN_NPARAM][n_sets], set-minor */
  const int32_t *set_of_env; /* device: [N] */
  int32_t n_sets, _pad;
} MdgParamSets;

/* mdg_step, mdg_step_autoreset, mdg_reset_ws and mdg_init_state with parameter sets.  NULL sets or n_sets < 1:
 * MDG_E_INVALID; a SINE* asset: MDG_E_UNSUPPORTED.  mdg_reset_ws_sets requires a workspace (NULL: MDG_E_INVALID).
 * The step kernel of these launches always runs in 128-thread blocks. */
int mdg_step_sets(const MdgParams *params, const MdgReward *reward, const MdgState *state, const MdgStepIO *io,
                  const MdgLaunch *launch, const MdgParamSets *sets);
int mdg_step_autoreset_sets(const MdgParams *params, const MdgReward *reward, const MdgState *state,
                            const MdgStepIO *io, const MdgLaunch *launch, int fill_ticks, int clear_nstep,
                            void *workspace, int64_t workspace_bytes, const MdgParamSets *sets);
int mdg_reset_ws_sets(const MdgParams *params, const MdgState *state, const MdgStepIO *io, const MdgLaunch *launch,
                      const uint8_t *mask, int fill_ticks, int clear_nstep, void *workspace, int64_t workspace_bytes,
                      const MdgParamSets *sets);
int mdg_init_state_sets(const MdgParams *params, const MdgReward *reward, const MdgState *state,
                        const MdgLaunch *launch, const MdgParamSets *sets);

/* ---------------------------------------------------------------------------------------------------
 * Broker sets: the seven broker settings of MdgParams per parameter set, so that the envs of one slab also trade under
 * different frictions (costs, slippage, margins, starting cash).
 *
 * The broker table is device memory [MDG_BROKER_NPARAM][n_sets], set-minor like MdgParamSets.p:
 * broker[k * n_sets + s] is slot k (MdgBrokerSlot, MdgParams field order) of set s.  It is indexed by the same
 * sets->set_of_env, with the same unsigned clamp to n_sets - 1.  With a broker table, every read of one of the seven
 * MdgParams fields by the step, refill, constructor and derived-accounting kernels reads the env's entry instead, and
 * the step kernel's risk-gate constants are computed per env with the same expressions as from MdgParams.  So env e
 * of such a launch is bit for bit env e of a launch without sets whose MdgParams hold the generator slots and the
 * broker settings of set s.  The values are not range-checked (neither are the MdgParams fields): any value, NaN
 * included, behaves per env as the same value does in MdgParams.  The table is read by each launch on its stream, as
 * the parameter-set table is.
 * broker == NULL: exactly the corresponding _sets launch (mdg_derived_sets_broker: mdg_derived).  NULL sets or
 * n_sets < 1: MDG_E_INVALID; a SINE* asset: MDG_E_UNSUPPORTED; mdg_reset_ws_sets_broker requires a workspace. */
enum MdgBrokerSlot {
  MDG_BROKER_INIT_CASH = 0,
  MDG_BROKER_REQUIRED_MARGIN = 1,
  MDG_BROKER_MAINTENANCE_MARGIN = 2,
  MDG_BROKER_SLIPPAGE_REL = 3,
  MDG_BROKER_SLIPPAGE_ABS = 4,
  MDG_BROKER_TCOST_REL = 5,
  MDG_BROKER_TCOST_ABS = 6
};
int mdg_step_sets_broker(const MdgParams *params, const MdgReward *reward, const MdgState *state,
                         const MdgStepIO *io, const MdgLaunch *launch, const MdgParamSets *sets, const double *broker);
int mdg_step_autoreset_sets_broker(const MdgParams *params, const MdgReward *reward, const MdgState *state,
                                   const MdgStepIO *io, const MdgLaunch *launch, int fill_ticks, int clear_nstep,
                                   void *workspace, int64_t workspace_bytes, const MdgParamSets *sets,
                                   const double *broker);
int mdg_reset_ws_sets_broker(const MdgParams *params, const MdgState *state, const MdgStepIO *io,
                             const MdgLaunch *launch, const uint8_t *mask, int fill_ticks, int clear_nstep,
                             void *workspace, int64_t workspace_bytes, const MdgParamSets *sets, const double *broker);
int mdg_init_state_sets_broker(const MdgParams *params, const MdgReward *reward, const MdgState *state,
                               const MdgLaunch *launch, const MdgParamSets *sets, const double *broker);

/* ---------------------------------------------------------------------------------------------------
 * Per-episode set draw: every refill of a listed env draws the env's parameter set anew (a new market per episode,
 * for training that is robust to the market), inside the launches a training loop already makes.
 *
 * cdf holds n_sets doubles (n_sets of the call's MdgParamSets): the cumulative sums of the weights, left to right,
 * over their total, with cdf[n_sets - 1] == 1.0 exactly; a set of weight 0 repeats its predecessor's entry and is never
 * drawn.  The draw of env e at tick t takes Philox4x32-10 with key (seed lo, seed hi) and counter
 * (env_offset + e, 4 << 16, t lo, t hi), x0 = (out[1] << 32) | out[0], u = (x0 >> 11) 2^-53, and yields the number
 * of cdf entries <= u (clamped to n_sets - 1).  It depends on (seed, global env id, tick, cdf) only, and uses Philox
 * also when the normals / uniforms are injected.
 *   - Refill (mdg_reset_ws_sets_draw, mdg_step_autoreset_sets_draw, both refill kernels): t is the env's timestamp
 *     before the refill; the refill writes episode_set[e] = the set the env had (clamped as the kernels read it) and
 *     set_of_env[e] = the drawn set, and runs the new episode (generator restart, history ticks, starting cash) in
 *     the drawn set.  Every refill advances the timestamp, so no two draws of one env share a counter.
 *   - Constructor (mdg_init_state_sets_draw): t = 0; it writes set_of_env[e] before the start values and the starting
 *     cash are read, and episode_set[e] = -1 (no episode has finished).
 * So these launches WRITE sets->set_of_env.  The step kernel is unchanged: it reads the set the refill left.
 * draw == NULL: exactly the corresponding _sets_broker launch (broker may be NULL: the _sets launch).  A draw whose
 * cdf or episode_set is NULL: MDG_E_INVALID; otherwise the checks of the _sets_broker launches. */
typedef struct MdgSetDraw {
  const double *cdf;    /* device: [n_sets] */
  int32_t *episode_set; /* device: [N], written for each listed env */
} MdgSetDraw;
int mdg_step_autoreset_sets_draw(const MdgParams *params, const MdgReward *reward, const MdgState *state,
                                 const MdgStepIO *io, const MdgLaunch *launch, int fill_ticks, int clear_nstep,
                                 void *workspace, int64_t workspace_bytes, const MdgParamSets *sets,
                                 const double *broker, const MdgSetDraw *draw);
int mdg_reset_ws_sets_draw(const MdgParams *params, const MdgState *state, const MdgStepIO *io,
                           const MdgLaunch *launch, const uint8_t *mask, int fill_ticks, int clear_nstep,
                           void *workspace, int64_t workspace_bytes, const MdgParamSets *sets, const double *broker,
                           const MdgSetDraw *draw);
int mdg_init_state_sets_draw(const MdgParams *params, const MdgReward *reward, const MdgState *state,
                             const MdgLaunch *launch, const MdgParamSets *sets, const double *broker,
                             const MdgSetDraw *draw);

/* Recompute MdgState.folds from the state tensors (after external writes into them). */
int mdg_refresh_folds(const MdgParams *params, const MdgState *state, const MdgLaunch *launch);

/* Portfolio's derived accounting for every env. */
int mdg_derived(const MdgParams *params, const MdgState *state, const MdgDerived *out,
                const MdgLaunch *launch);
/* ... with broker sets: required_margin and maintenance_margin of every env from its set (see MdgBrokerSlot) */
int mdg_derived_sets_broker(const MdgParams *params, const MdgState *state, const MdgDerived *out,
                            const MdgLaunch *launch, const MdgParamSets *sets, const double *broker);

/* StackerDiscrete.current_data price window (preprocessor.py:183-189) with the
 * normalisers of preprocessor.py:53-107: ring [k][F][N] -> out (N,k,F) or (N,F,k).
 * n_valid = rows currently in the window (<= k), oldest first. */
typedef struct MdgWindow {
  const double *ring;        /* [k][F][N] obs_price or obs_port                               */
  const double *prefix;      /* [N][k][F] pre_price, or NULL                                   */
  const int64_t *timestamp;  /* [N] MdgState.timestamp (NULL: every row comes from the ring)   */
  const int64_t *reset_ts;   /* [N] MdgState.reset_ts                                          */
  int64_t n_envs;
  int32_t n_feats, window, head, n_valid;
  int32_t norm_type;         /* MDG_NORM_*                                                     */
  int32_t flat_prefix;       /* prefix==NULL and rows older than the reset are [1,0,...,0]     */
  int32_t out_dtype, out_layout;
  void *out;                 /* (N, n_valid, F_out) or (N, F_out, n_valid)                    */
  void *stream;
  int32_t transform;         /* MDG_XFORM_*: the other price stackers of utils/preprocessor.py */
  int32_t stride;            /* MultiStackerDiscrete (preprocessor.py:202-288): window row s is the ring row of age
                                age0 + (n_valid-1-s) * stride; 0 or 1 = every row                                */
  int32_t age0;              /* age of the newest window row (0 = the newest ring row)                          */
  int32_t out_feats_total;   /* > 0: `out` has this many features per row and this window goes to columns
                                [out_feat_offset, out_feat_offset + F_out) -- the concatenation over dilations  */
  int32_t out_feat_offset;
  int32_t _pad;
} MdgWindow;
#define MDG_XFORM_NONE 0       /* StackerDiscrete            preprocessor.py:143-199, F_out = F            */
#define MDG_XFORM_PAIR_RATIO 1 /* StackerDiscretePairs       :295-321  price[:,0]/price[:,1], F = 2 -> F_out = 1, then the normaliser */
#define MDG_XFORM_RETURNS 2    /* StackerDiscreteReturns     :324-333  normaliser, then np.diff over the LAST axis
                                  (features, as the reference does): F_out = F - 1 */
int mdg_materialise_window(const MdgWindow *w);
/* (N, n_valid) int64 timestamps of the window rows: timestamp[e] - (n_valid-1-s) */
int mdg_materialise_time(const int64_t *timestamp, int64_t n_envs, int32_t n_valid, int64_t *out, void *stream);

/* Reduce the slab to MDG_STATS_NSCALAR + 2*nA doubles (per-asset sum |position value|/equity
 * and count of non-flat positions): the vector that is all-reduced across GPUs. */
int mdg_episode_stats(const MdgParams *params, const MdgState *state, const MdgStepIO *io,
                      const MdgLaunch *launch, double *out /* device, zeroed by the call */);

/* ---------------------------------------------------------------------------------------------------
 * Device-side n-step replay ingest (SURVEY section 8f rank 1): ReplayBuffer.add + NStepBuffer.pop_nstep_sarsd
 * (utils/buffers/replay_buffer.py:68-92, nstep_buffer.py:336-361) for every env of the slab, and
 * ReplayBuffer._sample (replay_buffer.py:110-132) as a gather -- observations never leave HBM.
 *
 * Observations are stored ONCE per step: obs slot t % depth holds, for every env, the window an agent sees after
 * step t ((N,k,F) as written by mdg_materialise_window, plus the newest portfolio row).  A transition is a record
 * (env, slot of its state, slot of its next_state, action, n-step shaped reward, done) in a global ring; the
 * step kernel has already produced the popped rewards (io.shaped_reward / io.n_popped) with the reference's
 * full-buffer / drain-on-done semantics, so the pops of step t are
 *     state = obs[t - L], action = a[t - L + 1], next_state = obs[t], done = done[t],  L = len, len-1, ...
 * Deviation (documented): with auto-reset the window of a finished env is materialised after its reset, so the
 * next_state of a terminal transition is the first observation of the next episode (the bootstrap is masked by
 * `done`); that same slot is, correctly, the state of the next episode's first transition. */
typedef struct MdgReplay {
  /* transition ring, capacity `capacity` records, structure of arrays */
  int32_t *t_env, *t_state_slot, *t_next_slot; /* [capacity] */
  int64_t *t_state_step;                       /* [capacity] step index of the state's observation (staleness check) */
  uint8_t *t_done;                             /* [capacity] */
  double *t_reward;                            /* [capacity][ra] */
  double *t_action;                            /* [capacity][n_action] */
  unsigned long long *cursor;                  /* [1] transitions appended so far (monotonic) */
  double *act_ring;                            /* [nstep][N][n_action] actions of the last nstep steps */
  int64_t capacity;
  int32_t depth;                               /* observation slots */
  int32_t nstep, ra, n_action;
} MdgReplay;

/* After step `step` (0-based count of agent steps of this slab): records `action` (N, n_action) and appends the
 * transitions popped by that step.  nstep_len = MdgState.nstep_len AFTER the step (NULL when nstep == 1). */
int mdg_replay_append(const MdgReplay *rp, int64_t n_envs, int64_t step, const double *action,
                      const double *shaped_reward /* [nstep][ra][N] */, const int32_t *n_popped,
                      const int32_t *nstep_len, const uint8_t *done, void *stream);

/* Draw `batch` transition indices uniformly from the stored, non-stale transitions (Philox keyed by seed, draw)
 * and gather the batch.  obs_price: [depth][N][k*F] (dtype out_dtype), obs_port: [depth][N][n_port] f64.
 * Outputs (device): idx [batch] int64, state/next price (batch, k*F), state/next portfolio row (batch, n_port),
 * action (batch, n_action), reward (batch, ra), done (batch) uint8. */
typedef struct MdgReplayBatch {
  int64_t *idx;
  void *state_price, *next_price;
  double *state_port, *next_port, *action, *reward;
  uint8_t *done;
} MdgReplayBatch;
int mdg_replay_sample(const MdgReplay *rp, int64_t n_envs, int64_t cur_step, const void *obs_price,
                      const double *obs_port, int32_t window_elems, int32_t n_port, int32_t obs_dtype,
                      int64_t batch, uint64_t seed, uint64_t draw, const MdgReplayBatch *out, void *stream);

/* ---------------------------------------------------------------------------------------------------
 * Proportional prioritized replay over the ring of MdgReplay (Schaul et al. 2016, the segment-tree form of the
 * reference's PrioritizedReplayBuffer, utils/buffers/prioritized_replay_buffer.py + segment_tree.py).
 *
 * A sum tree and a min tree in heap layout over the ring's slots: node 1 is the root, node j has the children 2j and
 * 2j+1, the leaf of ring slot i is node tree_size + i (tree_size: a power of two >= max(capacity, 1024)).  Every
 * internal node is left + right (min(left, right)), recomputed from its two children, so a tree is a pure function of
 * its leaves.  An unfilled leaf is 0 in the sum tree and +inf in the min tree.
 *   ingest  every record appended since the last ingest takes the leaf max_priority ** alpha (max_priority starts at
 *           1); a slot the ring overwrites takes the new record's priority.
 *   sample  total = sum root, seg = total / batch.  Sample b draws u (Philox, below) and descends with the mass
 *           u * seg + b * seg: at each node, go left if the left child > mass, else subtract it and go right.  A leaf
 *           that is unfilled, has priority 0, or is stale (its state's observation slot was overwritten, the test of
 *           mdg_replay_sample) is rejected and redrawn from the whole distribution (mass u * total, a fresh draw);
 *           after 64 attempts the row is idx = -1, position -1, weight 0, a zero row with done = 1.
 *           weight = (p_i / total * n) ** -beta / (p_min / total * n) ** -beta, n = filled records,
 *           p_min = the min root.
 *   update  applies to the batch of the last sample, in batch order as a sequential loop would: idx = -1 is
 *           skipped; so is a record the ring overwrote since it was sampled (leaf_pos differs from the sampled
 *           position); a priority that is not finite or not > 0 is skipped and counted in n_rejected; otherwise the
 *           leaf becomes priority ** alpha and max_priority = max(max_priority, priority).  Of an index that appears
 *           twice, the last occurrence wins.
 * Philox: sample b, attempt a uses the counter (b lo, (b hi) ^ (a << 8) ^ 0x80000000, draw lo, draw hi) with the
 * key seed, u = (x0 >> 11) 2^-53; bit 31 of the second word keeps these draws apart from mdg_replay_sample's.
 * Deviation (documented): a stale leaf keeps its mass until the ring overwrites it.  Rejection keeps sampling exactly
 * proportional over the resident records, but the weights' total and p_min include the stale leaves.
 * Every call enqueues a fixed number of launches with grids known to the host and never synchronises, so ingest,
 * sample and update can be captured in a CUDA graph.  Trees are rebuilt per 1024-leaf subtree: the calls that change
 * leaves list the subtrees they touch, one refresh kernel rebuilds the listed ones and its last block the levels
 * above them. */
typedef struct MdgPrioritized {
  double *sum_tree, *min_tree;   /* [2 * tree_size], node 0 unused */
  int64_t *leaf_pos;             /* [capacity] cursor position of the record in each slot, -1 = unfilled */
  int32_t *batch_pos;            /* [capacity] mdg_per_update scratch (last batch position per leaf), -1 between calls */
  uint32_t *dirty;               /* [tree_size / 1024] subtree marks, 0 between calls */
  int32_t *dirty_list;           /* [tree_size / 1024] the marked subtrees */
  uint32_t *ctl;                 /* [4] marked count, refresh exit ticket, ingest exit ticket, unused: zero before the
                                    first call, left zero by every call */
  unsigned long long *seen;      /* [1] MdgReplay.cursor as of the last ingest, 0 at first */
  double *max_priority;          /* [1] 1.0 at first */
  unsigned long long *n_rejected;/* [1] priorities update skipped as not finite or not > 0 */
  int64_t capacity;              /* == MdgReplay.capacity */
  int64_t tree_size;
  double alpha;
} MdgPrioritized;

/* After mdg_replay_append on the same stream (PrioritizedReplayBuffer.add): leaves of the records appended since
 * the last call.  max_new: a bound on their count (n_envs * nstep), sizes the grid. */
int mdg_per_ingest(const MdgPrioritized *pr, const MdgReplay *rp, int64_t max_new, void *stream);
/* PrioritizedReplayBuffer.sample: the arguments and the gather of mdg_replay_sample, plus weights [batch] f64 and the
 * sampled records' cursor positions pos [batch] int64 (what mdg_per_update checks against overwrites). */
int mdg_per_sample(const MdgPrioritized *pr, const MdgReplay *rp, int64_t n_envs, int64_t cur_step,
                   const void *obs_price, const double *obs_port, int32_t window_elems, int32_t n_port,
                   int32_t obs_dtype, int64_t batch, double beta, uint64_t seed, uint64_t draw,
                   const MdgReplayBatch *out, double *weights, int64_t *pos, void *stream);
/* PrioritizedReplayBuffer.update_priorities for the batch of the last sample: idx and pos as mdg_per_sample wrote
 * them, priorities [batch] f64. */
int mdg_per_update(const MdgPrioritized *pr, int64_t batch, const int64_t *idx, const int64_t *pos,
                   const double *priorities, void *stream);

/* ---------------------------------------------------------------------------------------------------
 * Replay row store: the observations of MdgReplay kept as raw price rows instead of materialised windows, and the
 * windows built and normalised at sample time for the sampled records only.
 *
 * Storage (device):
 *   rows       [N][n_rows][n_feats] f64, env-major: a per-env ring of raw price rows.  Rows are counted from 1:
 *              env e has appended row_count[e] rows, and row c is at position c % n_rows.
 *   row_count  [N] int64, rows appended per env (monotonic, 0 at first)
 *   row_end    [depth][N] int64: for observation slot t % depth, row_count[e] right after step t's ingest (0 = never
 *              written).  The window of that observation is the rows row_end - k + 1 ... row_end, oldest first.
 *   last_ts    [N] int64, the env's timestamp at its last ingest
 * Invariant: the k rows that end at row_end[t % depth][e] are bit for bit the raw (k, F) window mdg_materialise_window
 * (norm NONE, f64, n_valid = k) writes for env e after step t.
 * Ingest rule (mdg_replay_rows_ingest), per env, with since = timestamp - reset_ts + 1 and the rows read as
 * mdg_materialise_window reads them (ring rows for ages < since, prefix rows otherwise):
 *   - whole_window != 0, since == 1 (the env reset at this observation) or timestamp != last_ts + 1: append the whole
 *     k-row window (a reset's history fill, or whatever the window holds after a fill shorter than k);
 *   - otherwise append one row, the newest ring row (at `head`).
 * Timestamps are monotone across resets (reset_ts = timestamp + fill), so the rule covers auto-reset, explicit resets
 * between the step and the ingest, and fills shorter than k.  An env-step costs one row; a reset k rows.
 * Residency: a record is drawn only when the test of mdg_replay_sample holds AND its state's rows are still in the
 * ring:  row_end >= k  and  row_end - k + 1 > row_count - n_rows  (row_end of the state's slot).  The next state's
 * rows are newer.  Every reset during a record's life costs k - 1 extra rows, so with
 * n_rows >= depth + (k - 1)(r + 1) no record of an env that reset at most r times in `depth` steps goes stale through
 * its rows; n_rows < depth + k - 1 is rejected.  The Philox counters and draw loops are those of mdg_replay_sample and
 * mdg_per_sample, so when no record is stale through its rows both samplers draw the same indices as with stored
 * windows, and the batches are bit-identical to theirs (the windows are normalised by the same device code as
 * mdg_materialise_window's).
 * Deviation (documented), prioritized: a record stale through its rows keeps its leaf's mass until the ring overwrites
 * it, like a record whose observation slot was overwritten; the weights' total and p_min include it. */
typedef struct MdgReplayRows {
  double *rows;         /* [N][n_rows][n_feats] */
  int64_t *row_end;     /* [depth][N] */
  int64_t *row_count;   /* [N] */
  int64_t *last_ts;     /* [N] */
  int64_t n_rows;       /* rows kept per env */
  int32_t n_feats;      /* F, the env's assets */
  int32_t window;       /* k, the env's window */
} MdgReplayRows;

/* After a step (or for the first observation, with whole_window = 1): the ingest rule above for every env, reading the
 * env's observation ring through w (ring = obs_price, prefix = pre_price, timestamp, reset_ts, head, window, n_envs,
 * n_feats, stream; n_valid must equal window), then row_end[slot] = row_count.  slot in [0, depth). */
int mdg_replay_rows_ingest(const MdgReplayRows *rows, const MdgWindow *w, int64_t slot, int32_t whole_window);
/* mdg_replay_sample over the row store: windows normalised with norm_type (MDG_NORM_*) and written as out_dtype
 * (MDG_DTYPE_*), (batch, k, F); the other outputs as mdg_replay_sample. */
int mdg_replay_sample_rows(const MdgReplay *rp, const MdgReplayRows *rows, int64_t n_envs, int64_t cur_step,
                           const double *obs_port, int32_t n_port, int32_t norm_type, int32_t out_dtype,
                           int64_t batch, uint64_t seed, uint64_t draw, const MdgReplayBatch *out, void *stream);
/* mdg_per_sample over the row store (windows as mdg_replay_sample_rows). */
int mdg_per_sample_rows(const MdgPrioritized *pr, const MdgReplay *rp, const MdgReplayRows *rows, int64_t n_envs,
                        int64_t cur_step, const double *obs_port, int32_t n_port, int32_t norm_type,
                        int32_t out_dtype, int64_t batch, double beta, uint64_t seed, uint64_t draw,
                        const MdgReplayBatch *out, double *weights, int64_t *pos, void *stream);

/* ---------------------------------------------------------------------------------------------------
 * Streaming reward normalisers (environments/reward_normalization.pyx:14-272): one scalar state machine per env,
 * fed one raw reward (a log return) per step.  Every pointer is [N] (the queue storage [window][N]).
 *   SHARPE_FIXED   :61-118   reward / rolling std (Welford add at the head, remove at the tail), min 2 samples
 *   SORTINO_A      :121-145  the same, negative outputs squared in magnitude
 *   SORTINO_B / C  :148-218  std over the below-mean rewards only (B squares negative outputs, C does not)
 *   SHARPE_EWMA    :221-272  reward / exponentially weighted std, alpha = 2 / (window + 1)
 *   NULL           :49-58    identity */
enum MdgRewardNormKind {
  MDG_RN_NULL = 0,
  MDG_RN_SHARPE_FIXED = 1,
  MDG_RN_SORTINO_A = 2,
  MDG_RN_SORTINO_B = 3,
  MDG_RN_SORTINO_C = 4,
  MDG_RN_SHARPE_EWMA = 5
};
typedef struct MdgRewardNorm {
  int32_t kind;
  int32_t window;
  int64_t n_envs;
  double alpha;     /* SHARPE_EWMA: 2 / (window + 1)                               */
  double *buffer;   /* [window][N] the queue (ring storage), fixed-window kinds     */
  int32_t *size;    /* [N] queue length                                             */
  int32_t *front;   /* [N] ring slot of the queue front                             */
  int32_t *count;   /* [N] SORTINO_B/C: samples in the estimate; SHARPE_EWMA: count */
  double *mean_est; /* [N]                                                          */
  double *ssq;      /* [N]                                                          */
  double *ewma, *ewma_old, *ewssq_old, *ewssq, *w1, *w2; /* [N] SHARPE_EWMA        */
} MdgRewardNorm;
/* reset(): empty queue and zero estimates for the envs with mask[e] != 0 (mask == NULL: all) */
int mdg_reward_norm_reset(const MdgRewardNorm *rn, const uint8_t *mask, void *stream);
/* out[e] = shaper_e.stream(reward[e]) for every env; envs with reset_mask[e] != 0 (nullable) are reset() first --
 * "needs to be called when environment resets / episode ends" (reward_normalization.pyx:84) */
int mdg_reward_norm_stream(const MdgRewardNorm *rn, const double *reward, const uint8_t *reset_mask, double *out,
                           void *stream);

/* ---------------------------------------------------------------------------------------------------
 * On-device episode tearsheet (utils/metrics.py:83-171 test_summary and its helpers :334-421): the reference
 * records every step of a test episode on the host (equity, reward, ledger, transaction costs) and reduces the
 * lists with pandas at the end; here every env streams its episode into a handful of accumulators, one kernel per
 * step, and one kernel turns them into the tearsheet fields.  An env accumulates while active[e] != 0; the step
 * that reports done[e] is the last one recorded (the reference's `while not done` loop), then the env is frozen
 * until mdg_tearsheet_reset re-arms it.  Call mdg_tearsheet_update AFTER the step and BEFORE the env is reset.
 * Returns are log returns of the equity curve at offsets 2^j steps, j < n_offsets (metrics.py:71-78,367-411 with unit
 * timestamps); std by Welford (the reference: two-pass numpy; results agree to ~1e-12).
 * Every pointer is [N] unless noted. */
#define MDG_TS_MAX_OFFSETS 8
typedef struct MdgTearsheet {
  int64_t n_envs;
  int32_t n_assets;
  int32_t n_offsets;       /* J: offsets 1, 2, 4, ..., 2^(J-1); eq_ring holds 2^(J-1) equities per env */
  int64_t *nsteps;
  uint8_t *active;
  double *sum_equity, *last_equity, *sum_reward, *peak, *min_valley, *sum_cost;
  double *in_pos;          /* [nA][N] steps with ledger != 0 */
  double *eq_ring;         /* [2^(J-1)][N] */
  int32_t *ret_n;          /* [J][N] valid returns */
  double *ret_mean, *ret_m2, *ret_down; /* [J][N] Welford mean / M2, sum of squared negative returns */
} MdgTearsheet;
/* fields of mdg_tearsheet_summary's output, [MDG_TS_NFIXED + 3*J + nA][N]:
 *   0 nsteps 1 mean_equity 2 final_equity 3 mean_reward 4 max_drawdown (min of equity / expanding max, metrics.py:413-421)
 *   5 mean_transaction_cost (over steps x assets) 6 total_transaction_cost
 *   7+3j equity_returns_offset_2^j (nanmean)  8+3j equity_sharpe_offset_2^j (:334-348)  9+3j equity_sortino_offset_2^j
 *   (:350-365); NaN when 2^j > (nsteps-1)//10 (:108,133)
 *   7+3J+a time_spent_in_pos_<asset a> (:116-122) */
#define MDG_TS_NFIXED 7
int mdg_tearsheet_reset(const MdgTearsheet *ts, const uint8_t *mask, void *stream);
int mdg_tearsheet_update(const MdgParams *params, const MdgState *state, const MdgStepIO *io, const MdgTearsheet *ts,
                         void *stream);
int mdg_tearsheet_summary(const MdgTearsheet *ts, double *out, void *stream);

/* ---------------------------------------------------------------------------------------------------
 * Episode results: an exact table with one row per parameter set, filled on the device over every episode a run ends.
 * Each recording step updates the tearsheet ts exactly as mdg_tearsheet_update does; for every env whose step reported
 * done it then takes the env's tearsheet row exactly as mdg_tearsheet_summary would produce it, divides the four
 * money fields (1 mean_equity, 2 final_equity, 5 mean_transaction_cost, 6 total_transaction_cost) by the episode's
 * starting cash (the init_cash slot of its broker set, else MdgParams.init_cash), adds the row into the row of the
 * episode's set (set_of_env[e] before the refill, clamped as the kernels clamp it; 0 without sets) and re-arms the env's
 * recorder as mdg_tearsheet_reset does.
 *
 * Quantisation: a field value v is admitted when it is finite and |v| < 2^31 (NaN, +-inf and larger values are not
 * counted: n_episodes - count says how many were left out).  X = rint(v 2^64) is an exact integer (for |v| >= 2^-11 it
 * is v 2^64 unrounded); its five base-2^30 two's-complement digits (the top one signed) are each added with an int64
 * atomic into a limb of their own.  v*v (one fp64 multiply) goes the same way into the sum-of-squares limbs.  min and
 * max are order-preserving int64 images of the fp64 value (b = its bits; b < 0 ? b ^ 0x7fff...f : b) under
 * atomicMin / atomicMax.  Integer addition is associative: the table does not depend on the order in which envs
 * finish, the grid or the number of shards, and shards reduce with a plain SUM of acc (MIN / MAX of ext).
 * A limb grows by less than 2^30 per episode: the owner normalises the digits (back to [0, 2^30), the top digit signed)
 * at least every floor(2^32 / n_envs) recording steps, so that no limb overflows.
 *
 * Layout (int64, device):
 *   acc [n_sets][2 + 11 n_fields]: n_episodes, n_margin_call (episodes whose last step had margin_call set), then per
 *       field f: count, sum digits 0..4 (digit k has weight 2^(30k - 64)), sum-of-squares digits 0..4;
 *       zero when empty.
 *   ext [2][n_sets][n_fields]: min images, then max images; INT64_MAX / INT64_MIN when empty.
 * n_fields == MDG_TS_NFIXED + 3 ts.n_offsets + ts.n_assets (the tearsheet fields, in mdg_tearsheet_summary's order);
 * n_sets == the call's sets->n_sets, 1 without sets. */
typedef struct MdgEpisodeResults {
  MdgTearsheet ts; /* the recorder */
  int64_t *acc;    /* [n_sets][2 + 11 n_fields] */
  int64_t *ext;    /* [2][n_sets][n_fields] */
  int32_t n_sets, n_fields;
} MdgEpisodeResults;
/* mdg_step_autoreset_sets_draw with the record + harvest kernel between the step kernel and the refill (three
 * launches).  sets, broker and draw may each be NULL: a plain Env (then broker and draw must be NULL), no broker table,
 * no draw.  res is required; MDG_E_INVALID for a null accumulator or table, an n_assets, n_fields or n_sets that does
 * not match, or null done / margin_call. */
int mdg_step_autoreset_results(const MdgParams *params, const MdgReward *reward, const MdgState *state,
                               const MdgStepIO *io, const MdgLaunch *launch, int fill_ticks, int clear_nstep,
                               void *workspace, int64_t workspace_bytes, const MdgParamSets *sets,
                               const double *broker, const MdgSetDraw *draw, const MdgEpisodeResults *res);
/* the record + harvest kernel alone, for a step whose finished envs are reset separately (injected noise): call it
 * after the step and before the reset. */
int mdg_episode_results_record(const MdgParams *params, const MdgState *state, const MdgStepIO *io,
                               const MdgParamSets *sets, const double *broker, const MdgEpisodeResults *res,
                               void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MADIGAN_B200_H_ */
