//! Raw bindings, one to one with `include/azb.h` (same order, same names).  `tests/test_rust_binding.py` checks the
//! struct layouts, the function list and the constants against the header and the ctypes binding.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

pub const AZB_VERSION: c_int = 100;
pub const AZB_NONE: u32 = 0xFFFF_FFFF;
pub const AZB_MAX_VERTICES: u32 = 64;
pub const AZB_MAX_TOL: usize = 8;
pub const AZB_CKPT_MAGIC: u64 = 0x3154_504B_4342_5A41; // "AZBCKPT1"
pub const AZB_CKPT_FORMAT: u32 = 1;
pub const AZB_CKPT_HEADER_WORDS: u32 = 96;
pub const AZB_ASYNC_AUTO: u32 = 0xFFFF_FFFF;

pub const AZB_OK: c_int = 0;
pub const AZB_ERR_INVALID: c_int = 1;
pub const AZB_ERR_CUDA: c_int = 2;
pub const AZB_ERR_CAPACITY: c_int = 3;
pub const AZB_ERR_NAN: c_int = 4;
pub const AZB_ERR_LAMBDA: c_int = 5;
pub const AZB_ERR_UNREACHABLE: c_int = 6;
pub const AZB_ERR_STATE: c_int = 7;

pub const AZB_PRIOR_MLP: u32 = 0;
pub const AZB_PRIOR_HASH: u32 = 1;
pub const AZB_PRIOR_INJECTED: u32 = 2;

pub const AZB_MLP_FP32: u32 = 0;
pub const AZB_MLP_TC: u32 = 1;
pub const AZB_MLP_TC3: u32 = 2;

pub const AZB_SELECT_REFERENCE: u32 = 0;
pub const AZB_SELECT_PUCT: u32 = 1;

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct azb_config {
    pub struct_size: u32,
    pub n_vertices: u32,
    pub n_roots: u32,
    pub device: i32,
    pub first_root: u64,
    pub c_lower: f32,
    pub c_upper: f32,
    pub n_as_tol: [u32; 8],
    pub n_as_tol_len: u32,
    pub n_as_tol_default: u32,
    pub mlp_hidden: [u32; 3],
    pub mlp_mode: u32,
    pub prior_mode: u32,
    pub prior_seed: u64,
    pub max_steps: u32,
    pub cap_nodes: u32,
    pub cap_preds: u32,
    pub cap_parents: u32,
    pub max_episodes: u32,
    pub n_groups: u32,
    pub async_workers: u32,
    pub selection: u32,
    pub puct_c: f32,
    pub reserved: [u32; 3],
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct azb_counters {
    pub n_sel: u64,
    pub d_sel: u64,
    pub n_cur: u64,
    pub n_cand: u64,
    pub n_probe: u64,
    pub n_ins: u64,
    pub n_term: u64,
    pub n_hit: u64,
    pub n_arc: u64,
    pub n_pred: u64,
    pub n_cn: u64,
    pub d_cn: u64,
    pub n_reset: u64,
    pub n_live: u64,
    pub n_noop: u64,
    pub n_visit: u64,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct azb_improvement {
    pub step: u32,
    pub tree: u32,
    pub node: u32,
    pub eval: f32,
}

#[repr(C)]
pub struct azb_handle {
    _private: [u8; 0],
}

extern "C" {
    pub fn azb_version() -> c_int;
    pub fn azb_strerror(code: c_int) -> *const c_char;
    pub fn azb_last_error(h: *const azb_handle) -> *const c_char;
    pub fn azb_config_default(cfg: *mut azb_config, n_vertices: u32, n_roots: u32) -> c_int;
    pub fn azb_create(cfg: *const azb_config, out: *mut *mut azb_handle) -> c_int;
    pub fn azb_destroy(h: *mut azb_handle) -> c_int;
    pub fn azb_get_config(h: *const azb_handle, out: *mut azb_config) -> c_int;
    pub fn azb_generate_roots(seed: u64, first_root: u64, count: u32, n_vertices: u32, k_min: u32, k_max: u32, parents: *mut u8, permitted: *mut u32) -> c_int;
    pub fn azb_set_roots(h: *mut azb_handle, parents: *const u8, permitted: *const u32) -> c_int;
    pub fn azb_get_roots(h: *mut azb_handle, parents: *mut u8, permitted: *mut u32) -> c_int;
    pub fn azb_mlp_num_params(h: *const azb_handle) -> usize;
    pub fn azb_mlp_init(h: *mut azb_handle, seed: u64) -> c_int;
    pub fn azb_mlp_set_params(h: *mut azb_handle, params: *const f32) -> c_int;
    pub fn azb_mlp_get_params(h: *mut azb_handle, params: *mut f32) -> c_int;
    pub fn azb_model_write_predictions(h: *mut azb_handle, states: *const f32, predictions: *mut f32, rows: u32) -> c_int;
    pub fn azb_set_priors(h: *mut azb_handle, priors: *const f32) -> c_int;
    pub fn azb_init_trees(h: *mut azb_handle) -> c_int;
    pub fn azb_step(h: *mut azb_handle, n_steps: u32, improvements: *mut azb_improvement, cap: u32, n_improved: *mut u32) -> c_int;
    pub fn azb_step_enqueue(h: *mut azb_handle, n_steps: u32) -> c_int;
    pub fn azb_step_poll(h: *mut azb_handle, out: *mut azb_improvement, improved: *mut c_int) -> c_int;
    pub fn azb_step_timed(h: *mut azb_handle, n_steps: u32, ms: *mut f32, n_improved: *mut u32) -> c_int;
    pub fn azb_step_profile(h: *mut azb_handle, n_steps: u32, tree_ms: *mut f32, mlp_ms: *mut f32) -> c_int;
    pub fn azb_rollout_host(h: *mut azb_handle, state_vecs: *mut f32) -> c_int;
    pub fn azb_add_actions_host(h: *mut azb_handle, h_theta: *const f32, improved: *mut c_int) -> c_int;
    pub fn azb_get_argmin(h: *mut azb_handle, parents: *mut u8, permitted: *mut u32, lambda1: *mut f64, mu: *mut u32, eval: *mut f32) -> c_int;
    pub fn azb_get_node_state(h: *mut azb_handle, tree: u32, node: u32, parents: *mut u8, permitted: *mut u32) -> c_int;
    pub fn azb_tree_codes(h: *mut azb_handle, parents: *const u8, m: u32, codes: *mut u64, ms: *mut f32) -> c_int;
    pub fn azb_best_trees(h: *mut azb_handle, k: u32, n_out: *mut u32, eval: *mut f32, codes: *mut u64, tree: *mut u32, node: *mut u32, parents: *mut u8, permitted: *mut u32, lambda1: *mut f64, mu: *mut u32) -> c_int;
    pub fn azb_free_tree_count(n: u32, count: *mut u64) -> c_int;
    pub fn azb_free_trees(h: *mut azb_handle, start: u64, m: u32, parents: *mut u8) -> c_int;
    pub fn azb_exhaustive_best(h: *mut azb_handle, start: u64, count: u64, k: u32, bound: f64, n_out: *mut u32, n_below: *mut u64, index: *mut u64, parents: *mut u8, lambda1: *mut f64, mu: *mut u32, eval: *mut f32, ms: *mut f32) -> c_int;
    pub fn azb_trees_within(h: *mut azb_handle, bound: f64, k: u32, max_level: u64, n_out: *mut u32, n_within: *mut u64, n_below: *mut u64, codes: *mut u64, parents: *mut u8, lambda1: *mut f64, mu: *mut u32, eval: *mut f32, ms: *mut f32) -> c_int;
    pub fn azb_trees_within_proof(h: *mut azb_handle, bound: f64, k: u32, max_level: u64, n_out: *mut u32, n_within: *mut u64, n_below: *mut u64, codes: *mut u64, parents: *mut u8, lambda1: *mut f64, mu: *mut u32, eval: *mut f32, proof: *mut u64, ms: *mut f32) -> c_int;
    pub fn azb_certify_keys(h: *mut azb_handle, parents: *const u8, m: u32, bound: f64, lambda1_lo: *mut f64, lambda1_hi: *mut f64, mu: *mut u32, verdict: *mut i8, ms: *mut f32) -> c_int;
    pub fn azb_comm_trees_within(h: *mut azb_handle, bound: f64, k: u32, max_level: u64, n_out: *mut u32, n_within: *mut u64, n_below: *mut u64, codes: *mut u64, parents: *mut u8, lambda1: *mut f64, mu: *mut u32, eval: *mut f32, ms: *mut f32) -> c_int;
    pub fn azb_checkpoint_size(h: *mut azb_handle, bytes: *mut u64) -> c_int;
    pub fn azb_checkpoint_save(h: *mut azb_handle, buf: *mut c_void, size: u64, written: *mut u64) -> c_int;
    pub fn azb_checkpoint_load(h: *mut azb_handle, blobs: *const *const c_void, sizes: *const u64, n_blobs: u32) -> c_int;
    pub fn azb_get_walkers(h: *mut azb_handle, parents: *mut u8, permitted: *mut u32, path: *mut u32, pos: *mut u32, path_len: *mut u32) -> c_int;
    pub fn azb_tree_sizes(h: *mut azb_handle, tree: u32, n_nodes: *mut u32, n_arcs: *mut u32, n_preds: *mut u32) -> c_int;
    pub fn azb_dump_tree(h: *mut azb_handle, tree: u32, nodes: *mut u32, keys: *mut u32, preds: *mut u32, arcs: *mut u32) -> c_int;
    pub fn azb_get_counters(h: *mut azb_handle, out: *mut azb_counters) -> c_int;
    pub fn azb_reset_counters(h: *mut azb_handle) -> c_int;
    pub fn azb_set_counter_mode(h: *mut azb_handle, full: c_int) -> c_int;
    pub fn azb_get_state_vecs(h: *mut azb_handle, state_vecs: *mut f32) -> c_int;
    pub fn azb_get_priors(h: *mut azb_handle, priors: *mut f32) -> c_int;
    pub fn azb_eval_costs(h: *mut azb_handle, parents: *const u8, m: u32, lambda1: *mut f64, mu: *mut u32, c: *mut f32, ms: *mut f32) -> c_int;
    pub fn azb_eval_graph_costs(h: *mut azb_handle, nbr: *const u32, m: u32, n: u32, lambda1: *mut f64, mu: *mut u32, kinds: *mut u32, ms: *mut f32) -> c_int;
    pub fn azb_eval_graph_costs64(h: *mut azb_handle, nbr: *const u64, m: u32, n: u32, lambda1: *mut f64, mu: *mut u32, kinds: *mut u32, ms: *mut f32) -> c_int;
    pub fn azb_write_observations(h: *mut azb_handle, n_obs_tol: u32, state_vecs: *mut f32, observations: *mut f32, weights: *mut f32) -> c_int;
    pub fn azb_adam_config(h: *mut azb_handle, lr: f32, beta1: f32, beta2: f32, eps: f32, l2: f32) -> c_int;
    pub fn azb_model_update(h: *mut azb_handle, states: *const f32, observations: *const f32, action_weights: *const f32, rows: u32, loss: *mut f32) -> c_int;
    pub fn azb_model_gradients(h: *mut azb_handle, states: *const f32, observations: *const f32, action_weights: *const f32, rows: u32, loss: *mut f32, grads: *mut f32) -> c_int;
    pub fn azb_update_model(h: *mut azb_handle, n_obs_tol: u32, loss: *mut f32) -> c_int;
    pub fn azb_reset_trees(h: *mut azb_handle, seed: u64, k_min: u32, k_max: u32) -> c_int;
    pub fn azb_comm_unique_id(id128: *mut u8) -> c_int;
    pub fn azb_comm_init(h: *mut azb_handle, id128: *const u8, rank: c_int, world: c_int) -> c_int;
    pub fn azb_comm_destroy(h: *mut azb_handle) -> c_int;
    pub fn azb_comm_allreduce_bench(h: *mut azb_handle, reps: u32, ms: *mut f32) -> c_int;
    pub fn azb_comm_argmin(h: *mut azb_handle, parents: *mut u8, permitted: *mut u32, lambda1: *mut f64, mu: *mut u32, eval: *mut f32, owner_rank: *mut c_int) -> c_int;
    pub fn azb_kernel_launches(h: *const azb_handle, n: *mut u64) -> c_int;
    pub fn azb_device_bytes(h: *const azb_handle, bytes: *mut u64) -> c_int;
    pub fn azb_flush_l2(h: *mut azb_handle) -> c_int;
    pub fn azb_debug_cascade_spills(h: *mut azb_handle, n: *mut u32) -> c_int;
}
