/*
 * ust.h — C ABI of libust.so, the B200-native per-node driver-upgrade state machine.
 *
 * One call to ust_apply_state*() evaluates, for every node of a cluster snapshot, the transition
 * that the reference's ClusterUpgradeStateManagerImpl.ApplyState() would make
 * (reference: pkg/upgrade/upgrade_state.go:171-281), on one B200 (or sharded over the B200s of one
 * NVSwitch box). The snapshot is a struct-of-arrays encoding of ClusterUpgradeState
 * (reference: pkg/upgrade/common_manager.go:58-80); the policy is a flat copy of
 * DriverUpgradePolicySpec (reference: api/upgrade/v1alpha1/upgrade_spec.go:27-110) plus the
 * manager options (reference: pkg/upgrade/upgrade_state.go:329-350, :94-96).
 *
 * The library never evaluates a node on the CPU: every entry point that computes fails with
 * UST_ERR_CUDA when no sm_100 device / kernel image is available.
 *
 * Plain C, no torch types: this header is what a cgo / ctypes / JNI binding binds (INTEGRATION.md).
 */
#ifndef UST_H_
#define UST_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UST_ABI_VERSION 1

/* ------------------------------------------------------------------------------------------------
 * Node upgrade-state codes — the value of the node label nvidia.com/<driver>-driver-upgrade-state
 * (reference: pkg/upgrade/consts.go:49-82, key format consts.go:21).
 * ---------------------------------------------------------------------------------------------- */
enum {
  UST_STATE_UNKNOWN = 0,                    /* ""                          consts.go:50 */
  UST_STATE_UPGRADE_REQUIRED = 1,           /* "upgrade-required"          consts.go:53 */
  UST_STATE_CORDON_REQUIRED = 2,            /* "cordon-required"           consts.go:55 */
  UST_STATE_WAIT_FOR_JOBS_REQUIRED = 3,     /* "wait-for-jobs-required"    consts.go:57 */
  UST_STATE_POD_DELETION_REQUIRED = 4,      /* "pod-deletion-required"     consts.go:59 */
  UST_STATE_DRAIN_REQUIRED = 5,             /* "drain-required"            consts.go:62 */
  UST_STATE_NODE_MAINTENANCE_REQUIRED = 6,  /* "node-maintenance-required" consts.go:67 */
  UST_STATE_POST_MAINTENANCE_REQUIRED = 7,  /* "post-maintenance-required" consts.go:71 */
  UST_STATE_POD_RESTART_REQUIRED = 8,       /* "pod-restart-required"      consts.go:74 */
  UST_STATE_VALIDATION_REQUIRED = 9,        /* "validation-required"       consts.go:77 */
  UST_STATE_UNCORDON_REQUIRED = 10,         /* "uncordon-required"         consts.go:79 */
  UST_STATE_DONE = 11,                      /* "upgrade-done"              consts.go:81 */
  UST_STATE_FAILED = 12,                    /* "upgrade-failed"            consts.go:83 */
  UST_STATE_OTHER = 13,    /* any other label value: bucketed by BuildState (upgrade_state.go:158-160),
                              counted by GetCurrentUnavailableNodes, never processed */
  UST_STATE_EXCLUDED = 14, /* driver pod with NodeName=="" && Phase==Pending: BuildState skips it
                              (upgrade_state.go:149-152) — not part of the snapshot */
  UST_NUM_STATE_CODES = 16 /* code 15 is reserved and treated like UST_STATE_EXCLUDED */
};

/* ------------------------------------------------------------------------------------------------
 * state[i] (uint8): the "hot" byte. Low nibble = state code above. High nibble = the four node
 * predicates the cluster-wide constraint logic needs: one shared-memory lookup indexed by this byte
 * gives the kernel a node's counter increments and its transition-table window, and the passes that
 * only count or rank (ordered slot allocation, pod-list selection, BuildState) read nothing else.
 * ---------------------------------------------------------------------------------------------- */
#define UST_HOT_STATE_MASK 0x0Fu
#define UST_HOT_NOT_READY 0x10u   /* some NodeReady condition has Status != True   common_manager.go:656-663 */
#define UST_HOT_SKIP 0x20u        /* label ...-driver-upgrade.skip == "true"       common_manager.go:666-668 */
#define UST_HOT_UNSCHEDULABLE 0x40u /* node.Spec.Unschedulable                     common_manager.go:651-653 */
#define UST_HOT_REVISION_HASH_ERROR 0x80u
/* ^ revision-hash lookup fails for a NON-orphaned driver pod: controller-revision-hash label absent
 *   (pod_manager.go:84-89) or no ControllerRevision for its DaemonSet (pod_manager.go:108-110).
 *   ApplyState aborts with an error when it reaches such a node in the unknown / upgrade-done /
 *   pod-restart-required / upgrade-failed passes (common_manager.go:234-238, :463-467, :533-538). */

/* ------------------------------------------------------------------------------------------------
 * flags[i] (uint32): one bit per reference predicate on the node / its driver pod.
 * Bits 0-4, 9, 10 and 22-31 are reserved for values the kernel derives itself (skip / unschedulable
 * from the hot byte, slot grant, pod-in-sync, pod-list summaries) and are ignored on input. The
 * positions are chosen so that the bits each state's transition reads are contiguous (the kernel
 * indexes a per-state table with a 9-bit window of this word).
 * ---------------------------------------------------------------------------------------------- */
#define UST_F_UPGRADE_REQUESTED (1u << 5)  /* annotation ...-driver-upgrade-requested == "true"  common_manager.go:323-325 */
#define UST_F_VALIDATION_DONE (1u << 6)    /* ValidationManager.Validate() == true               common_manager.go:587-596 */
#define UST_F_SAFE_LOAD (1u << 7)          /* annotation ...driver-wait-for-safe-load != ""      safe_driver_load_manager.go:51-53 */
#define UST_F_POD_ORPHANED (1u << 8)       /* DriverDaemonSet == nil                             common_manager.go:66-68 */
#define UST_F_POD_READY (1u << 11)         /* Phase==Running && len(ContainerStatuses)!=0 && all Ready   common_manager.go:617-630 */
#define UST_F_INITIAL_STATE_ANNO (1u << 12) /* annotation ...node-initial-state.unschedulable PRESENT    common_manager.go:545, :680 */
#define UST_F_REQUESTOR_MODE (1u << 13)    /* annotation ...-driver-upgrade-requestor-mode PRESENT       util.go:135-138 */
#define UST_F_POD_TERMINATING (1u << 14)   /* !DriverPod.DeletionTimestamp.IsZero()              common_manager.go:472 */
#define UST_F_POD_FAILING (1u << 15)       /* some (init)container !Ready && RestartCount > 10   common_manager.go:636-648 */
#define UST_F_WAIT_PODS_RUNNING (1u << 16) /* a wait-selector pod is Running or Pending          pod_manager.go:278-284, :371-391 */
#define UST_F_WAIT_START_ANNO (1u << 17)   /* annotation ...wait-for-pod-completion-start-time PRESENT   pod_manager.go:336 */
#define UST_F_WAIT_TIMED_OUT (1u << 18)    /* now > start + timeout                              pod_manager.go:354 */
#define UST_F_WAIT_START_INVALID (1u << 19) /* start-time annotation does not parse as int64     pod_manager.go:348-353 */
#define UST_F_NM_PRESENT (1u << 20)        /* NodeUpgradeState.NodeMaintenance != nil            upgrade_requestor.go:420 */
#define UST_F_NM_READY (1u << 21)          /* NodeMaintenance Ready condition with Reason Ready  upgrade_requestor.go:437-439 */
#define UST_F_INPUT_MASK 0x003FF9E0u

/* ------------------------------------------------------------------------------------------------
 * pod_flags[p] (uint16): one entry per workload pod of a node (CSR by pod_off), used to evaluate
 * what the asynchronous actuators would decide (kubectl drain filter chain, k8s.io/kubectl v0.35.1
 * pkg/drain/filters.go; call sites pod_manager.go:146-157,191 and drain_manager.go:76-96,121).
 * ---------------------------------------------------------------------------------------------- */
#define UST_POD_PHASE_MASK 0x0007u
enum { UST_PHASE_OTHER = 0, UST_PHASE_PENDING = 1, UST_PHASE_RUNNING = 2, UST_PHASE_SUCCEEDED = 3, UST_PHASE_FAILED = 4 };
#define UST_POD_HAS_CONTROLLER (1u << 3)       /* metav1.GetControllerOf(pod) != nil */
#define UST_POD_CONTROLLED_BY_DS (1u << 4)     /* ... and its Kind is DaemonSet */
#define UST_POD_DS_MISSING (1u << 5)           /* that DaemonSet cannot be fetched (NotFound) */
#define UST_POD_MIRROR (1u << 6)               /* kubernetes.io/config.mirror annotation present */
#define UST_POD_HAS_EMPTYDIR (1u << 7)         /* a volume with EmptyDir != nil */
#define UST_POD_MATCH_DELETION_FILTER (1u << 8) /* PodDeletionFilter(pod) == true     pod_manager.go:76,139,179 */
#define UST_POD_MATCH_WAIT_SELECTOR (1u << 9)  /* matches WaitForCompletionSpec.PodSelector   pod_manager.go:263 */
#define UST_POD_MATCH_DRAIN_SELECTOR (1u << 10) /* matches DrainSpec.PodSelector       drain_manager.go:86 */

/* ------------------------------------------------------------------------------------------------
 * actions[i] (uint16): the actuator / provider calls ApplyState makes for node i, in addition to the
 * label change implied by next_state[i] != state code. One bit per call site.
 * ---------------------------------------------------------------------------------------------- */
#define UST_A_SET_STATE (1u << 0)               /* ChangeNodeUpgradeState(next_state) */
#define UST_A_SET_INITIAL_STATE_ANNO (1u << 1)  /* common_manager.go:253-264 */
#define UST_A_CLEAR_INITIAL_STATE_ANNO (1u << 2) /* common_manager.go:558-565, :699-706 */
#define UST_A_CLEAR_UPGRADE_REQUESTED (1u << 3) /* upgrade_inplace.go:72-81, upgrade_requestor.go:285-294 */
#define UST_A_CORDON (1u << 4)                  /* common_manager.go:366 */
#define UST_A_UNCORDON (1u << 5)                /* upgrade_inplace.go:133 */
#define UST_A_SCHEDULE_WAIT_CHECK (1u << 6)     /* node passed to ScheduleCheckOnPodCompletion  common_manager.go:413-414 */
#define UST_A_SCHEDULE_POD_EVICTION (1u << 7)   /* node passed to SchedulePodEviction           common_manager.go:443-452 */
#define UST_A_SCHEDULE_DRAIN (1u << 8)          /* node passed to ScheduleNodesDrain            common_manager.go:350-356 */
#define UST_A_RESTART_DRIVER_POD (1u << 9)      /* pod passed to SchedulePodsRestart            common_manager.go:472-474, :523 */
#define UST_A_UNBLOCK_SAFE_LOAD (1u << 10)      /* safe_driver_load_manager.go:57-71 */
#define UST_A_SET_WAIT_START (1u << 11)         /* pod_manager.go:336-345 (actuator evaluation only) */
#define UST_A_CLEAR_WAIT_START (1u << 12)       /* pod_manager.go:301-302, :360 (actuator evaluation only) */
#define UST_A_REQUESTOR_ANNO_CHANGE (1u << 13)  /* upgrade_requestor.go:302-306 (set), :476-480 (clear) */
#define UST_A_NM_CREATE_OR_DELETE (1u << 14)    /* upgrade_requestor.go:296, :482 */
#define UST_A_ERROR (1u << 15)                  /* ApplyState returns an error at this node */

/* actuator_outcome[i] when no actuator runs for the node */
#define UST_OUTCOME_NONE 0xFFu

/* ------------------------------------------------------------------------------------------------
 * Policy: DriverUpgradePolicySpec (upgrade_spec.go:27-110) + manager options, flattened.
 * ---------------------------------------------------------------------------------------------- */
enum { UST_MAXUNAVAIL_NIL = 0, UST_MAXUNAVAIL_INT = 1, UST_MAXUNAVAIL_PERCENT = 2, UST_MAXUNAVAIL_INVALID = 3 };

typedef struct ust_policy {
  int32_t auto_upgrade;            /* AutoUpgrade; 0 => ApplyState is a successful no-op (upgrade_state.go:179-182) */
  int32_t max_unavailable_kind;    /* UST_MAXUNAVAIL_*: nil / intstr.Int / "NN%" / unparsable string */
  int64_t max_parallel_upgrades;   /* MaxParallelUpgrades; 0 = unlimited */
  int64_t max_unavailable_value;   /* IntVal, or NN of "NN%" */
  int32_t pod_deletion_enabled;    /* WithPodDeletionEnabled(filter != nil)      upgrade_state.go:329-337 */
  int32_t validation_enabled;      /* WithValidationEnabled(selector != "")      upgrade_state.go:341-350 */
  int32_t pod_deletion_spec_present; /* PodDeletion != nil */
  int32_t pod_deletion_force;      /* PodDeletionSpec.Force */
  int32_t pod_deletion_delete_emptydir; /* PodDeletionSpec.DeleteEmptyDir */
  int32_t drain_enabled;           /* DrainSpec != nil && DrainSpec.Enable       upgrade_state.go:235 */
  int32_t drain_force;             /* DrainSpec.Force */
  int32_t drain_delete_emptydir;   /* DrainSpec.DeleteEmptyDir */
  int32_t wait_selector_set;       /* WaitForCompletion != nil && PodSelector != ""   common_manager.go:392 */
  int32_t wait_timeout_nonzero;    /* WaitForCompletionSpec.TimeoutSecond != 0       pod_manager.go:290 */
  int32_t use_maintenance_operator; /* StateOptions.Requestor.UseMaintenanceOperator  upgrade_state.go:291,302,321 */
  int32_t evaluate_actuators;      /* 1: also fill actuator_outcome / wait-start actions from the
                                         WAIT_* flag bits and, when given, the pod lists */
} ust_policy;

/* ------------------------------------------------------------------------------------------------
 * Cluster-wide results of one call (what CommonUpgradeStateManager's getters return,
 * common_manager.go:715-788, plus the slot arithmetic of upgrade_inplace.go:49-62).
 * ---------------------------------------------------------------------------------------------- */
enum {
  UST_OK = 0,
  UST_ERR_INVALID_ARGUMENT = -1,
  UST_ERR_CUDA = -2,            /* no device, no sm_100 image, launch or copy failure */
  UST_ERR_NIL_STATE = -3,       /* "currentState should not be empty"           upgrade_state.go:175-177 */
  UST_ERR_REVISION_HASH = -4,   /* per-node abort, see UST_HOT_REVISION_HASH_ERROR */
  UST_ERR_MAX_UNAVAILABLE = -5, /* intstr.GetScaledValueFromIntOrPercent fails   upgrade_inplace.go:54-60 */
  UST_ERR_POD_DELETION_SPEC = -6, /* "pod deletion spec should not be empty"     pod_manager.go:132-134 */
  UST_ERR_DS_UNSCHEDULED = -7,  /* "driver DaemonSet should not have Unscheduled pods"  upgrade_state.go:128-131 */
  UST_ERR_COMM = -8,            /* multi-GPU exchange failed */
  UST_ERR_TRUNCATED = -9        /* ust_apply_state_delta_sparse: more changed outputs than the caller's arrays hold */
};

typedef struct ust_counters {
  int64_t hist[UST_NUM_STATE_CODES]; /* nodes per state code (index 14 = excluded entries) */
  int64_t unavailable;        /* GetCurrentUnavailableNodes               common_manager.go:146-165 */
  int64_t candidates;         /* upgrade-required nodes not marked skip */
  int64_t total_managed;      /* GetTotalManagedNodes                     common_manager.go:715-730 */
  int64_t in_progress;        /* GetUpgradesInProgress                    common_manager.go:733-739 */
  int64_t max_unavailable;    /* scaled MaxUnavailable                    upgrade_inplace.go:52-60 */
  int64_t upgrades_available; /* GetUpgradesAvailable (may be negative)   common_manager.go:748-776 */
  int64_t error_code;         /* UST_OK or the UST_ERR_* ApplyState aborted with */
  int64_t error_index;        /* node index it aborted at; -1 for a policy-level error */
  int64_t error_pass;         /* 0-based position of the aborting Process* pass in upgrade_state.go:205-274 */
  int64_t reserved[7];
} ust_counters;

/* Optional per-node workload pod lists (CSR). pod_off has n_nodes+1 entries; for device-resident calls
 * pod_flags must be 16-byte aligned like every other array (the list reader uses 16-byte loads, never past
 * pod_flags + n_pods). pod_off is int32: one call (one shard) holds fewer than 2^31 workload pods - at BASELINE's 30
 * pods per node that is 71 M nodes per GPU; shard further before that. The host entry points check the offsets
 * (pod_off[0] == 0, non-decreasing, pod_off[n_nodes] == n_pods => UST_ERR_INVALID_ARGUMENT otherwise);
 * ust_apply_state_device trusts the caller's device arrays. */
typedef struct ust_pods {
  const int32_t* pod_off;
  const uint16_t* pod_flags;
  int64_t n_pods;
} ust_pods;

typedef struct ust_handle ust_handle;

/* ---- lifetime ---------------------------------------------------------------------------------- */

/* Create a handle bound to CUDA device `device` (>= 0). The handle owns one stream, its staging
 * buffers (grown geometrically) and a 64 KiB workspace. Not re-entrant; distinct handles are
 * independent. Returns UST_OK or UST_ERR_CUDA (then *out == NULL). */
int ust_create(ust_handle** out, int device);
void ust_destroy(ust_handle* h);
/* Message for the last non-OK return on this handle (never NULL; valid until the next call). */
const char* ust_last_error(const ust_handle* h);
/* Same, for failures of ust_create itself (thread-local). */
const char* ust_create_error(void);
int ust_abi_version(void);
/* Number of kernels this handle has launched so far (for bench.py's gpu_launches). */
int64_t ust_launch_count(const ust_handle* h);

/* Pinned host memory for the SoA arrays (optional; pageable pointers also work, more slowly). */
void* ust_host_alloc(size_t bytes);
void ust_host_free(void* p);

/* ---- ApplyState -------------------------------------------------------------------------------- */

/* Replaces ClusterUpgradeStateManagerImpl.ApplyState (upgrade_state.go:171-281) for a snapshot given
 * as host arrays. All pointers are caller-owned and are not retained after return.
 *   policy == NULL or !auto_upgrade  => no-op: next_state = state code, actions = 0, returns UST_OK.
 *   n_nodes < 0 or NULL arrays       => UST_ERR_NIL_STATE / UST_ERR_INVALID_ARGUMENT.
 * On a reference-level abort (UST_ERR_REVISION_HASH, _MAX_UNAVAILABLE, _POD_DELETION_SPEC) the outputs
 * hold exactly what the reference had done before returning the error: nodes the sequential passes
 * had not reached are left untouched, the aborting node carries UST_A_ERROR. */
int ust_apply_state(ust_handle* h, const ust_policy* policy, int64_t n_nodes,
                    const uint8_t* state, const uint32_t* flags, const int32_t* pod_rev,
                    const int32_t* ds_idx, int32_t n_ds, const int32_t* ds_rev,
                    const ust_pods* pods /* nullable */,
                    uint8_t* next_state, uint16_t* actions, uint8_t* actuator_outcome /* nullable */,
                    ust_counters* out /* nullable */);

/* Same computation on arrays already resident in device memory (16-byte aligned), enqueued on the
 * handle's stream (or `stream`, a cudaStream_t, when non-NULL). Returns after the launch;
 * `out_device` (nullable) receives the counters in device memory. Use ust_sync() before reading. */
int ust_apply_state_device(ust_handle* h, const ust_policy* policy, int64_t n_nodes,
                           const uint8_t* state, const uint32_t* flags, const int32_t* pod_rev,
                           const int32_t* ds_idx, int32_t n_ds, const int32_t* ds_rev,
                           const ust_pods* pods /* nullable; device pointers inside */,
                           uint8_t* next_state, uint16_t* actions, uint8_t* actuator_outcome,
                           ust_counters* out_device, void* stream);
int ust_sync(ust_handle* h);
/* The handle's own CUDA stream (a cudaStream_t), the one calls with stream == NULL run on. It belongs to the library:
 * a caller may record events on it, wait for it and make it wait for events, but must not enqueue kernels or copies
 * that write a call's arrays on it (produce inputs on a stream of your own and pass that stream, or order the two
 * streams with an event) - for this reason:
 * Back-to-back ust_apply_state_device calls on this stream that share no buffer with one another except read-only
 * inputs (different snapshots, different output arrays - a batch of clusters, a sweep of what-if policies) overlap: a
 * call's streaming kernel starts as the previous call's runs out of work, and that call's decision (and multi-GPU
 * exchange) runs beside it. Calls that share an output or feed on the previous call's outputs, calls with pod lists
 * and calls on any other stream keep the strict order. Results are the same either way. */
void* ust_stream(ust_handle* h);

/* Packed host format: ust_apply_state with the two interned columns at the width they need - pod_rev16[i] is the
 * interned driver-pod revision hash (0 = none) as uint16, ds_idx8[i] the DaemonSet index as int8 (< 0 = orphaned),
 * so 8 instead of 13 bytes per node cross PCIe; the device widens them. For encoders that intern at most 65535
 * revision hashes and 127 DaemonSets (the reference's driver DaemonSets per cluster are a handful); anything else
 * uses ust_apply_state. No pod lists. Same outputs, counters, errors and resident snapshot as ust_apply_state. */
int ust_apply_state_packed(ust_handle* h, const ust_policy* policy, int64_t n_nodes, const uint8_t* state,
                           const uint32_t* flags, const uint16_t* pod_rev16, const int8_t* ds_idx8, int32_t n_ds,
                           const int32_t* ds_rev, uint8_t* next_state, uint16_t* actions, uint8_t* actuator_outcome,
                           ust_counters* out);

/* Delta form (SURVEY 8f.2): a ust_apply_state without pod lists that succeeds or ends in a reference-level abort
 * (UST_ERR_REVISION_HASH, _MAX_UNAVAILABLE, _POD_DELETION_SPEC) leaves the uploaded snapshot resident on
 * the device. ust_apply_state_delta overwrites the n_changed nodes named by idx (distinct indices into that
 * snapshot) with freshly encoded values - what a reconcile that watches resourceVersions re-encodes - and evaluates
 * the whole snapshot again: same outputs and counters as ust_apply_state on the updated arrays, without
 * re-uploading the unchanged nodes. The DaemonSet table is passed in full (it is small). Returns
 * UST_ERR_INVALID_ARGUMENT when there is no resident snapshot (first call, a call with pod lists, or
 * ust_build_state* since, which share the staging memory). */
int ust_apply_state_delta(ust_handle* h, const ust_policy* policy, int64_t n_changed, const int64_t* idx,
                          const uint8_t* state, const uint32_t* flags, const int32_t* pod_rev, const int32_t* ds_idx,
                          int32_t n_ds, const int32_t* ds_rev, uint8_t* next_state, uint16_t* actions,
                          uint8_t* actuator_outcome, ust_counters* out);

/* Delta in, delta out: ust_apply_state_delta with sparse outputs. The previous call on this handle (ust_apply_state,
 * _packed, _delta or _delta_sparse - whose full next_state / actions the caller still holds) left its outputs on the
 * device; this call returns only the nodes whose (next_state, actions) differ from them, in node order:
 * out_idx[k], out_next_state[k], out_actions[k] for k < *n_out. Patching the caller's arrays with them gives exactly what
 * ust_apply_state_delta would have written - a reconcile with 1 % churn moves ~1 % of the 3 bytes per node back over
 * PCIe instead of all of them. When more than max_out outputs changed, *n_out holds the count, nothing is written to
 * the out_* arrays and UST_ERR_TRUNCATED is returned: fetch everything with ust_fetch_outputs. No actuator_outcome.
 * Reference-level aborts are reported like in ust_apply_state_delta (the sparse outputs are still delivered). */
int ust_apply_state_delta_sparse(ust_handle* h, const ust_policy* policy, int64_t n_changed, const int64_t* idx,
                                 const uint8_t* state, const uint32_t* flags, const int32_t* pod_rev, const int32_t* ds_idx,
                                 int32_t n_ds, const int32_t* ds_rev, int64_t max_out, int64_t* out_idx,
                                 uint8_t* out_next_state, uint16_t* out_actions, int64_t* n_out, ust_counters* out);
/* The full outputs of the last call on the resident snapshot (n_nodes entries each). */
int ust_fetch_outputs(ust_handle* h, uint8_t* next_state, uint16_t* actions);

/* Rollout simulation (SURVEY 8f.3) on the resident snapshot (see ust_apply_state_delta): `steps` reconciles in a row,
 * entirely on the device. After each ApplyState the decisions are fed back into the snapshot under "ideal
 * actuators": every provider call takes effect (state label, annotations, cordon / uncordon), every scheduled
 * asynchronous actuator succeeds with the state in actuator_outcome (evaluate_actuators is forced on), a restarted
 * driver pod comes back at its DaemonSet's current revision and ready (an orphaned one is gone: the node leaves the
 * snapshot), and what a node is still waiting for (jobs, pod readiness, validation) has happened by the next
 * reconcile - so the only thing that paces the rollout is the MaxParallelUpgrades / MaxUnavailable budget, which is
 * the planning question. history[k] (nullable, `steps` entries) receives the counters of reconcile k; final_*
 * (nullable) the snapshot afterwards; *steps_done the number of reconciles fed back. A reconcile that returns a
 * reference-level error stops the feedback: its code is returned, the state before it is kept. One GPU, no pod
 * lists; in-place and requestor mode (see ust_simulate_rollout_timed for what the maintenance operator is taken to do). */
int ust_simulate_rollout(ust_handle* h, const ust_policy* policy, int32_t steps, ust_counters* history,
                         uint8_t* final_state, uint32_t* final_flags, int32_t* final_pod_rev, int32_t* steps_done);

/* The same simulation with a clock: reconcile k runs at simulated time k * seconds_per_reconcile, and the things a
 * node waits for take time instead of having happened by the next reconcile. Per node the device keeps the time it
 * entered its state, its wait-for-pod-completion start time (the annotation of pod_manager.go:336-345) and its
 * validation start time (validation_manager.go:139-175):
 *   wait-for-jobs-required  the wait-selector pods of a node run until job_seconds after the node entered the state
 *                           (nodes already there at time 0: from time 0, if their UST_F_WAIT_PODS_RUNNING is set). While
 *                           they run: no start annotation => it is set to `now`; present and now > start +
 *                           wait_timeout_seconds => pod-deletion-required, annotation removed (pod_manager.go:331-368;
 *                           the policy's wait_timeout_nonzero must say whether wait_timeout_seconds != 0).
 *   validation-required     the validation pod is ready validation_seconds after the node entered the state (< 0: never).
 *                           Until then Validate() runs handleTimeout: no start annotation => set to `now`; present and
 *                           now > start + validation_timeout_seconds (600 in the reference, validation_manager.go:32) =>
 *                           upgrade-failed, annotation removed.
 *   requestor mode (policy->use_maintenance_operator, accepted by both simulation entry points): an upgrade-required
 *                           node gets its NodeMaintenance and the requestor-mode annotation (upgrade_requestor.go:277-319);
 *                           the maintenance operator cordons it and reports Ready maintenance_seconds after the object
 *                           was created (=> pod-restart-required, :416-452); the uncordon pass removes annotation and
 *                           object, the maintenance operator uncordons (:454-488).
 * With every field 0 (validation_timeout_seconds aside) this is ust_simulate_rollout. */
typedef struct ust_sim_options {
  int64_t seconds_per_reconcile;
  int64_t wait_timeout_seconds;
  int64_t job_seconds;
  int64_t validation_seconds;
  int64_t validation_timeout_seconds;
  int64_t maintenance_seconds;
} ust_sim_options;
int ust_simulate_rollout_timed(ust_handle* h, const ust_policy* policy, const ust_sim_options* options, int32_t steps,
                               ust_counters* history, uint8_t* final_state, uint32_t* final_flags, int32_t* final_pod_rev,
                               int32_t* steps_done);

/* ---- BuildState -------------------------------------------------------------------------------- */

/* The device part of BuildState (upgrade_state.go:99-164): per-DaemonSet count of owned driver pods
 * against DesiredNumberScheduled (:128-131, counted before the pending-skip of :149-152) and the
 * bucket sizes. One entry per driver pod; ds_idx < 0 = orphaned pod. Returns UST_ERR_DS_UNSCHEDULED
 * when some DaemonSet's count differs (counters->error_index = that DaemonSet's index). */
int ust_build_state(ust_handle* h, int64_t n_pods, const uint8_t* state, const int32_t* ds_idx,
                    int32_t n_ds, const int32_t* ds_desired, ust_counters* out);

/* The same with the owner join done on the device (upgrade_state.go:126-147, common_manager.go:168-227):
 * owner_uid holds, per driver pod, the 128-bit UID of OwnerReferences[0] as two uint64 (both 0 = the pod has no
 * owner reference: IsOrphanedPod, common_manager.go:225-227); ds_uid holds the UIDs of the driver DaemonSets
 * (the keys of GetDriverDaemonSets' map, so they must be distinct - UST_ERR_INVALID_ARGUMENT otherwise).
 * ds_idx_out[i] receives the index of the owning DaemonSet, -1 for an orphaned pod, -2 for a pod owned by
 * something else: GetPodsOwnedbyDs skips it and GetOrphanedPods does not take it, so it is not part of the
 * snapshot and not counted in any bucket (it shows up in hist[14], "not in snapshot"). Everything else as
 * ust_build_state; host arrays, no alignment requirement. */
int ust_build_state_uids(ust_handle* h, int64_t n_pods, const uint8_t* state, const uint64_t* owner_uid,
                         int32_t n_ds, const uint64_t* ds_uid, const int32_t* ds_desired, int32_t* ds_idx_out,
                         ust_counters* out);

/* ---- introspection ----------------------------------------------------------------------------- */

/* The kernel evaluates a node by one lookup in a per-policy table indexed by (state code, 9-bit window
 * of the node's predicate word w = flags | derived bits). These two calls expose that table (host side,
 * no device needed) so that it can be audited entry by entry:
 *   ust_table_entry: bits 0-15 actions, 16-23 next state, 24-31 actuator outcome (0xFF = none) for a
 *   node in state `state_code` whose predicate word is `w` (only the bits of the state's window matter);
 *   ust_table_window_shift: first bit of the window that state reads. */
uint32_t ust_table_entry(const ust_policy* policy, unsigned state_code, uint32_t w);
int ust_table_window_shift(unsigned state_code);

/* ---- multi-GPU (one process per GPU) ----------------------------------------------------------- */

#define UST_UNIQUE_ID_BYTES 128
/* Rank 0 calls ust_get_unique_id and distributes the bytes; every rank then calls ust_comm_init.
 * Nodes are sharded in contiguous index ranges, rank r before rank r+1 (slice order of the
 * upgrade-required bucket, upgrade_inplace.go:71, is global index order). Afterwards every
 * ust_apply_state* call is collective: each rank passes its shard and one exchange of the
 * constraint counters happens per call. */
int ust_get_unique_id(void* out_bytes);
int ust_comm_init(ust_handle* h, int rank, int world_size, const void* unique_id_bytes);
/* exchange mode: 0 = ncclAllReduce between two kernels (default), 1 = fused: each rank runs ONE kernel that pushes
 * its counters into every peer's mailbox over NVLink (CUDA IPC peer memory) and reads the peers' from its own.
 * Mode 1 returns UST_ERR_COMM when the peer mailboxes could not be mapped at ust_comm_init. All ranks must use the
 * same mode. */
int ust_comm_set_mode(ust_handle* h, int mode);

#ifdef __cplusplus
}
#endif
#endif /* UST_H_ */
