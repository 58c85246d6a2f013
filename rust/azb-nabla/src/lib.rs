//! `B200Optimizer`: the c21 example's `NablaOptimizer` (az-discrete-opt/src/nabla/optimizer/mod.rs:7-363) with the
//! batched search step running on a B200 through `libazb.so`.
//!
//! Same method names, argument meaning and return types as the reference, over the reference's own types
//! (`NablaModel`, `ROTWithActionPermissions<N>`, `Conjecture2Dot1Cost`, `ArgminData`, `ArgminImprovement`,
//! `ActionSet`), so `graph-state/examples/04-c21-tree.rs` changes in one line (`NablaOptimizer::par_new` ->
//! `B200Optimizer::par_new`); see `examples/c21.rs`.
//!
//! What crosses the boundary as DATA because closures cannot cross a C ABI: `N`, `C_LOWER_BOUND`/`C_UPPER_BOUND`
//! (04-c21-tree.rs:58-68), the `n_as_tol` table (`:136-138`).  Hard-wired in the kernels: `g = c_s - h`,
//! `h_sa = c*_as`, cost = lambda_1 + mu (`:96-105`).  `par_new` probes the space's function pointers on two states and
//! `par_roll_out_episodes` probes `n_as_tol` on depths 0..16, and both panic on a mismatch — like the reference, which
//! has no error returns on this path (optimizer/mod.rs:121-191; `panic = 'abort'`).
//!
//! Not compiled in the build image (no Rust toolchain): see rust/README.md for what is checked instead.
#![feature(isqrt)]

use std::{collections::BTreeSet, ffi::CStr, os::raw::{c_int, c_void}};

use az_discrete_opt::{
    log::ArgminData,
    nabla::{model::NablaModel, optimizer::ArgminImprovement, space::NablaStateActionSpace},
    path::{set::ActionSet, ActionPath},
};
use azb_sys as sys;
use graph_state::{
    rooted_tree::{
        modify_parent_once::ROTWithActionPermissions, ordered_edge::OrderedEdge, space::ROTModifyParentsOnce,
        RootedOrderedTree,
    },
    simple_graph::{connected_bitset_graph::Conjecture2Dot1Cost, edge::Edge},
};

pub type State<const N: usize> = ROTWithActionPermissions<N>;
pub type Cost = Conjecture2Dot1Cost;
pub type Space<const N: usize> = ROTModifyParentsOnce<N, Cost>;

/// ACTION_DIM and the number of 32-bit words of an action mask (rooted_tree/space.rs:46-48)
pub const fn action_dim(n: usize) -> usize {
    (n - 1) * (n - 2) / 2 - 1
}
pub const fn mask_words(n: usize) -> usize {
    (action_dim(n) + 31) / 32
}

/// Where `h_theta` comes from.
pub enum Model<M> {
    /// any `NablaModel` on the host: the reference's data flow, the two rayon regions replaced by two launches
    /// (`azb_rollout_host` / `azb_add_actions_host`), state vectors and predictions cross PCIe every step
    Host(M),
    /// the built-in MLP (the example's 2A-512-1024-512-A, `04-c21-tree.rs:46-52`): parameters in dfdx order
    /// (per `Linear`: `weight[out][in]` then `bias[out]`); nothing leaves the GPU inside an epoch
    Device { params: Vec<f32>, tensor_cores: bool },
}

/// The selection rule at an active node (`azb_config.selection`).
#[derive(Clone, Copy, Debug, PartialEq)]
pub enum Selection {
    /// the reference's `next_action` (`nabla/tree/next_action.rs:11-26`)
    Reference,
    /// PUCT with constant `c_puct` (finite, > 0); the rule is this library's own (`include/azb.h`) and has no
    /// reference to check it against
    Puct { c_puct: f32 },
}

/// The only two things the example's `modify_root` reads from a `StateWeight` (whose constructor is `pub(crate)`):
/// `c()` and `c_star()` (`nabla/tree/state_weight.rs:23-29`).
#[derive(Clone, Copy, Debug)]
pub struct NodeWeight {
    c: f32,
    c_star: f32,
}
impl NodeWeight {
    pub fn c(&self) -> f32 {
        self.c
    }
    pub fn c_star(&self) -> f32 {
        self.c_star
    }
}

pub struct B200Optimizer<const N: usize, M> {
    h: *mut sys::azb_handle,
    space: Space<N>,
    model: Option<M>, // None: device model
    batch: usize,
    roots: Vec<State<N>>,
    state_vecs: Vec<f32>,
    h_theta_host: Vec<f32>,
    action_weights: Vec<f32>,
    argmin_data: ArgminData<State<N>, Cost>,
    n_as_tol: [u32; 9], // the table the handle was created with: depths 0..8 and the default
    enqueued: u32,      // steps enqueued by roll_out_ahead that have not been polled yet
    reset_seed: u64,
}

// The handle is bound to one CUDA device and is not thread-safe; it may move between threads like `&mut self`.
unsafe impl<const N: usize, M: Send> Send for B200Optimizer<N, M> {}

fn last_error(h: *const sys::azb_handle, rc: c_int) -> String {
    unsafe {
        let what = CStr::from_ptr(sys::azb_strerror(rc)).to_string_lossy().into_owned();
        let detail = if h.is_null() { String::new() } else { CStr::from_ptr(sys::azb_last_error(h)).to_string_lossy().into_owned() };
        format!("azb error {rc} ({what}): {detail}")
    }
}

/// panics with the library's message: the reference's hot path has no error returns either (NaN, lambda_1 < 1.4 and
/// the unreachable branch all abort there: next_action.rs:51, ordered_edge.rs:79, tree/mod.rs:227)
fn ck(h: *const sys::azb_handle, rc: c_int) {
    if rc != sys::AZB_OK {
        panic!("{}", last_error(h, rc));
    }
}

/// `ROTWithActionPermissions<N>` -> (parents as bytes, permitted-action bit mask).  `RootedOrderedTree::parents` is
/// `pub(crate)`, so the parents of children 2..N-2 are read back from the public edge-index iterator
/// (rooted_tree/mod.rs:60-72); parents[1] and parents[N-1] are 0 for every state this space generates
/// (rooted_tree/mod.rs:14-20), and act() never touches them (actions are edges of children 2..N-2).
/// One isomorphism class of `best_trees`: its value, the representative node's state and cost, the canonical code
/// (include/azb.h) and where the representative lives (local tree, node).
pub struct BestTree<const N: usize> {
    pub eval: f32,
    pub lambda_1: f64,
    pub mu: u32,
    pub state: State<N>,
    pub code: [u64; 2],
    pub tree: u32,
    pub node: u32,
}

pub fn flatten<const N: usize>(s: &State<N>, parents: &mut [u8], permitted: &mut [u32]) {
    assert!(parents.len() == N && permitted.len() == mask_words(N));
    parents.fill(0);
    permitted.fill(0);
    for (i, e) in s.tree.edge_indices_ignoring_0_1_and_last_vertex().enumerate() {
        let edge = OrderedEdge::from_index_ignoring_edge_0_1(e);
        debug_assert_eq!(edge.child(), i + 2);
        parents[edge.child()] = edge.parent() as u8;
    }
    for &a in &s.permitted_actions {
        permitted[a / 32] |= 1u32 << (a % 32);
    }
}

pub fn unflatten<const N: usize>(parents: &[u8], permitted: &[u32]) -> State<N> {
    let mut p = [0usize; N];
    for i in 0..N {
        p[i] = parents[i] as usize;
    }
    let tree = RootedOrderedTree::<N>::try_from(p).expect("libazb returned an invalid parent array");
    let mut permitted_actions = BTreeSet::new();
    for a in 0..action_dim(N) {
        if permitted[a / 32] >> (a % 32) & 1 == 1 {
            permitted_actions.insert(a);
        }
    }
    ROTWithActionPermissions { tree, permitted_actions }
}

/// A `Conjecture2Dot1Cost` from (lambda_1, mu).  The library reports the matching NUMBER (all the reference's
/// `evaluate` and tensorboard summary read is `matching.len()`: 04-c21-tree.rs:99, connected_bitset_graph/mod.rs:358-363);
/// `with_matching = true` recomputes the edge list on the host with the reference's own routine.
fn cost_of<const N: usize>(state: &State<N>, lambda_1: f64, mu: u32, with_matching: bool) -> Cost {
    if with_matching {
        let c = state.tree.conjecture_2_1_cost();
        debug_assert_eq!(c.matching.len(), mu as usize);
        c
    } else {
        Conjecture2Dot1Cost { matching: vec![Edge::new(0, 1); mu as usize], lambda_1 }
    }
}

impl<const N: usize, M: NablaModel> B200Optimizer<N, M> {
    const A: usize = action_dim(N);
    const W: usize = mask_words(N);
    const S: usize = 2 * action_dim(N);

    /// `NablaOptimizer::par_new` (optimizer/mod.rs:39-118): `init_states` is called `batch` times on the host, the
    /// states are flattened and uploaded once, the library computes root costs, root vectors, one prior evaluation,
    /// root nodes and root predictions, and the silent argmin over the roots.
    /// `n_as_tol` is the closure the example later passes to `par_roll_out_episodes` (04-c21-tree.rs:136-138): the
    /// revisit budgets are part of the device configuration, so they are sampled here.
    pub fn par_new(
        space: Space<N>,
        init_states: impl Fn() -> State<N> + Sync + Send,
        model: Model<M>,
        batch: usize,
        n_as_tol: impl Fn(usize) -> u32,
        max_steps_per_epoch: u32,
    ) -> Self {
        Self::par_new_with_selection(space, init_states, model, batch, n_as_tol, max_steps_per_epoch, Selection::Reference)
    }

    /// `par_new` with a choice of selection rule (`Selection::Reference` is `par_new`).
    pub fn par_new_with_selection(
        space: Space<N>,
        init_states: impl Fn() -> State<N> + Sync + Send,
        model: Model<M>,
        batch: usize,
        n_as_tol: impl Fn(usize) -> u32,
        max_steps_per_epoch: u32,
        selection: Selection,
    ) -> Self {
        let roots: Vec<State<N>> = (0..batch).map(|_| init_states()).collect();
        let mut me = Self::with_handle(space, model, roots, n_as_tol, max_steps_per_epoch, selection, 0);
        me.assert_space_is_c21();
        me.upload_roots_and_init();
        me.refresh_argmin(true);
        me
    }

    /// Continue a saved run (azb_checkpoint_load): a handle over `batch` roots from global root `first_root`, loaded
    /// from the blobs of every rank of the saving run (any number of ranks).  Roots, trees, walkers, the device model
    /// and its Adam state, the running best and the reset count are the saved ones; a host model keeps its own state.
    /// The space, `n_as_tol` and `selection` must be the saving run's (the load refuses a different configuration).
    pub fn resume(
        space: Space<N>,
        model: Model<M>,
        batch: usize,
        first_root: u64,
        n_as_tol: impl Fn(usize) -> u32,
        max_steps_per_epoch: u32,
        selection: Selection,
        blobs: &[&[u8]],
    ) -> Self {
        assert!(!blobs.is_empty() && blobs[0].len() >= 8 * sys::AZB_CKPT_HEADER_WORDS as usize, "checkpoint blobs");
        let roots: Vec<State<N>> = (0..batch).map(|_| unflatten::<N>(&[0u8; N], &vec![0u32; Self::W])).collect();
        let mut me = Self::with_handle(space, model, roots, n_as_tol, max_steps_per_epoch, selection, first_root);
        let ptrs: Vec<*const c_void> = blobs.iter().map(|b| b.as_ptr() as *const c_void).collect();
        let sizes: Vec<u64> = blobs.iter().map(|b| b.len() as u64).collect();
        ck(me.h, unsafe { sys::azb_checkpoint_load(me.h, ptrs.as_ptr(), sizes.as_ptr(), blobs.len() as u32) });
        // the device reset seeds continue from the saved reset count (header word 28, include/azb.h)
        let resets = u64::from_le_bytes(blobs[0][8 * 28..8 * 29].try_into().unwrap());
        for _ in 0..resets {
            me.reset_seed = me.reset_seed.wrapping_mul(0x9E37_79B9_7F4A_7C15).wrapping_add(1);
        }
        let mut parents = vec![0u8; batch * N];
        let mut masks = vec![0u32; batch * Self::W];
        ck(me.h, unsafe { sys::azb_get_roots(me.h, parents.as_mut_ptr(), masks.as_mut_ptr()) });
        for (i, r) in me.roots.iter_mut().enumerate() {
            *r = unflatten::<N>(&parents[i * N..(i + 1) * N], &masks[i * Self::W..(i + 1) * Self::W]);
        }
        me.assert_space_is_c21();
        me.refresh_argmin(true);
        me
    }

    /// The search and training state as a checkpoint blob (azb_checkpoint_save; format in include/azb.h), after the
    /// steps `roll_out_ahead` enqueued have completed.
    pub fn save_checkpoint(&mut self) -> Vec<u8> {
        if self.enqueued > 0 {
            self.finish_batch();
        }
        let mut size = 0u64;
        ck(self.h, unsafe { sys::azb_checkpoint_size(self.h, &mut size) });
        let mut blob = vec![0u8; size as usize];
        let mut written = 0u64;
        ck(self.h, unsafe { sys::azb_checkpoint_save(self.h, blob.as_mut_ptr() as *mut c_void, size, &mut written) });
        blob.truncate(written as usize);
        blob
    }

    fn with_handle(
        space: Space<N>,
        model: Model<M>,
        roots: Vec<State<N>>,
        n_as_tol: impl Fn(usize) -> u32,
        max_steps_per_epoch: u32,
        selection: Selection,
        first_root: u64,
    ) -> Self {
        let batch = roots.len();
        assert!(N >= 5 && N <= sys::AZB_MAX_VERTICES as usize && batch > 0);
        let mut cfg: sys::azb_config = unsafe { std::mem::zeroed() };
        ck(std::ptr::null(), unsafe { sys::azb_config_default(&mut cfg, N as u32, batch as u32) });
        // the n_as_tol closure as a table: depths 0..8 explicit, the value at depth 8 as the default
        let mut table = [0u32; 9];
        for (d, t) in table.iter_mut().enumerate() {
            *t = n_as_tol(d);
        }
        cfg.n_as_tol.copy_from_slice(&table[..8]);
        cfg.n_as_tol_len = 8;
        cfg.n_as_tol_default = table[8];
        cfg.max_steps = max_steps_per_epoch;
        cfg.first_root = first_root;
        if let Selection::Puct { c_puct } = selection {
            cfg.selection = sys::AZB_SELECT_PUCT;
            cfg.puct_c = c_puct;
        }
        let (host_model, params) = match model {
            Model::Host(m) => {
                cfg.prior_mode = sys::AZB_PRIOR_INJECTED;
                (Some(m), None)
            }
            Model::Device { params, tensor_cores } => {
                cfg.prior_mode = sys::AZB_PRIOR_MLP;
                cfg.mlp_mode = if tensor_cores { sys::AZB_MLP_TC } else { sys::AZB_MLP_FP32 };
                // the asynchronous kernel wherever it applies; the library picks the model SMs for the root count
                cfg.async_workers = if tensor_cores { sys::AZB_ASYNC_AUTO } else { 0 };
                (None, Some(params))
            }
        };
        let mut h: *mut sys::azb_handle = std::ptr::null_mut();
        let rc = unsafe { sys::azb_create(&cfg, &mut h) };
        if rc != sys::AZB_OK {
            let msg = last_error(h, rc);
            unsafe { sys::azb_destroy(h) };
            panic!("{msg}");
        }
        if let Some(p) = &params {
            assert_eq!(p.len(), unsafe { sys::azb_mlp_num_params(h) }, "parameter block: dfdx order, weight[out][in] then bias[out] per Linear");
            ck(h, unsafe { sys::azb_mlp_set_params(h, p.as_ptr()) });
        }

        Self {
            h,
            space,
            model: host_model,
            batch,
            roots,
            state_vecs: vec![0.; batch * Self::S],
            h_theta_host: vec![0.; batch * Self::A],
            action_weights: vec![0.; batch * Self::A],
            argmin_data: ArgminData::new(unflatten::<N>(&[0u8; N], &vec![0u32; Self::W]), Conjecture2Dot1Cost::default(), f32::INFINITY),
            n_as_tol: table,
            enqueued: 0,
            reset_seed: 0x5EED,
        }
    }

    /// The kernels hard-wire the c21 closures; refuse any other space (two probe states, bit-exact f32).
    fn assert_space_is_c21(&self) {
        let probes = [&self.roots[0], &self.roots[self.batch - 1]];
        let mut parents = vec![0u8; 2 * N];
        let mut mask = vec![0u32; Self::W];
        for (i, s) in probes.iter().enumerate() {
            flatten::<N>(s, &mut parents[i * N..(i + 1) * N], &mut mask);
        }
        let (mut l1, mut mu, mut c) = ([0f64; 2], [0u32; 2], [0f32; 2]);
        ck(self.h, unsafe { sys::azb_eval_costs(self.h, parents.as_ptr(), 2, l1.as_mut_ptr(), mu.as_mut_ptr(), c.as_mut_ptr(), std::ptr::null_mut()) });
        for (i, s) in probes.iter().enumerate() {
            let cost = self.space.cost(s);
            assert_eq!(cost.matching.len(), mu[i] as usize, "space.cost is not the c21 cost");
            assert!((cost.lambda_1 - l1[i]).abs() <= 1e-9 * l1[i], "space.cost is not the c21 cost");
            assert_eq!(self.space.evaluate(&cost).to_bits(), c[i].to_bits(), "space.evaluate is not squish(mu + lambda_1) with the library's bounds");
        }
        assert_eq!(self.space.g_theta_star_sa(0.75, (), 0.25), 0.5, "g_theta_star_sa must be c_s - h");
        assert_eq!(self.space.h_sa(0.1, 0.2, 0.3), 0.3, "h_sa must be c*_as");
    }

    fn upload_roots_and_init(&mut self) {
        let mut parents = vec![0u8; self.batch * N];
        let mut masks = vec![0u32; self.batch * Self::W];
        for (i, s) in self.roots.iter().enumerate() {
            flatten::<N>(s, &mut parents[i * N..(i + 1) * N], &mut masks[i * Self::W..(i + 1) * Self::W]);
        }
        ck(self.h, unsafe { sys::azb_set_roots(self.h, parents.as_ptr(), masks.as_ptr()) });
        if let Some(m) = self.model.as_mut() {
            // the one model call of par_new / par_reset_trees (optimizer/mod.rs:69-71, 347-348) on the root vectors
            for (s, v) in self.roots.iter().zip(self.state_vecs.chunks_exact_mut(Self::S)) {
                self.space.write_vec(s, v);
            }
            self.h_theta_host.fill(0.);
            m.write_predictions(&self.state_vecs, &mut self.h_theta_host);
            ck(self.h, unsafe { sys::azb_set_priors(self.h, self.h_theta_host.as_ptr()) });
        }
        ck(self.h, unsafe { sys::azb_init_trees(self.h) });
        self.enqueued = 0;
    }

    /// `ArgminData { state, cost, eval }` from the library (optimizer/mod.rs:224-242 rebuilds the state by replaying
    /// the winning node's action set on its root; the device does the same replay: azb_get_argmin)
    fn refresh_argmin(&mut self, with_matching: bool) {
        let mut parents = vec![0u8; N];
        let mut mask = vec![0u32; Self::W];
        let (mut l1, mut mu, mut eval) = (0f64, 0u32, 0f32);
        ck(self.h, unsafe { sys::azb_get_argmin(self.h, parents.as_mut_ptr(), mask.as_mut_ptr(), &mut l1, &mut mu, &mut eval) });
        let state = unflatten::<N>(&parents, &mask);
        let cost = cost_of::<N>(&state, l1, mu, with_matching);
        self.argmin_data = ArgminData::new(state, cost, eval);
    }

    fn check_tol(&self, n_as_tol: &impl Fn(usize) -> u32) {
        for d in 0..16 {
            assert_eq!(n_as_tol(d), self.n_as_tol[d.min(8)], "n_as_tol({d}) differs from the table par_new sampled");
        }
    }

    pub fn get_model_mut(&mut self) -> Option<&mut M> {
        self.model.as_mut()
    }

    /// `par_roll_out_episodes` (optimizer/mod.rs:121-191), one step per call.
    /// Host model: rollout_host -> model.write_predictions -> add_actions_host (+ par_update_argmmim_data).
    /// Device model: steps enqueued by [`roll_out_ahead`] are reported one per call as soon as every tree has
    /// finished them (later steps keep running); without a prior `roll_out_ahead` the call is one blocking step.
    pub fn par_roll_out_episodes(&mut self, n_as_tol: impl Fn(usize) -> u32 + Sync) -> ArgminImprovement<State<N>, Cost> {
        self.check_tol(&n_as_tol);
        let mut improved: c_int = 0;
        if let Some(m) = self.model.as_mut() {
            ck(self.h, unsafe { sys::azb_rollout_host(self.h, self.state_vecs.as_mut_ptr()) });
            m.write_predictions(&self.state_vecs, &mut self.h_theta_host);
            ck(self.h, unsafe { sys::azb_add_actions_host(self.h, self.h_theta_host.as_ptr(), &mut improved) });
        } else if self.enqueued > 0 {
            let mut rec = sys::azb_improvement::default();
            ck(self.h, unsafe { sys::azb_step_poll(self.h, &mut rec, &mut improved) });
            self.enqueued -= 1;
            if improved != 0 {
                // ArgminData of the improving step while later steps still run, exactly like optimizer/mod.rs:224-242:
                // the tree's root with the node's action set replayed (azb_get_node_state), then the space's own cost
                // and evaluate on the host
                let mut parents = vec![0u8; N];
                let mut mask = vec![0u32; Self::W];
                ck(self.h, unsafe { sys::azb_get_node_state(self.h, rec.tree, rec.node, parents.as_mut_ptr(), mask.as_mut_ptr()) });
                let state = unflatten::<N>(&parents, &mask);
                let cost = self.space.cost(&state);
                let eval = self.space.evaluate(&cost);
                debug_assert_eq!(eval.to_bits(), rec.eval.to_bits());
                self.argmin_data = ArgminData::new(state, cost, eval);
            }
            if self.enqueued == 0 {
                self.finish_batch(); // device-side argmin state, improvement log and error check of the whole batch
            }
            return if improved != 0 { ArgminImprovement::Improved(&self.argmin_data) } else { ArgminImprovement::Unchanged };
        } else {
            let mut n: u32 = 0;
            let mut rec = sys::azb_improvement::default();
            ck(self.h, unsafe { sys::azb_step(self.h, 1, &mut rec, 1, &mut n) });
            improved = (n > 0) as c_int;
        }
        if improved != 0 {
            self.refresh_argmin(true);
            ArgminImprovement::Improved(&self.argmin_data)
        } else {
            ArgminImprovement::Unchanged
        }
    }

    /// Device model only: start `episodes` steps without waiting.  The example's loop (`for episode in 1..=episodes
    /// { optimizer.par_roll_out_episodes(n_as_tol) }`, 04-c21-tree.rs:142-143) then advances at the speed of the
    /// fused loop instead of one launch + synchronisation per step.
    pub fn roll_out_ahead(&mut self, episodes: u32) {
        assert!(self.model.is_none(), "roll_out_ahead needs the device model");
        assert_eq!(self.enqueued, 0, "the previous batch has unreported steps");
        ck(self.h, unsafe { sys::azb_step_enqueue(self.h, episodes) });
        self.enqueued = episodes;
    }

    /// azb_step(h, 0): waits for the enqueued steps, runs the device-side argmin pass, reports errors
    fn finish_batch(&mut self) {
        let mut n: u32 = 0;
        ck(self.h, unsafe { sys::azb_step(self.h, 0, std::ptr::null_mut(), 0, &mut n) });
        self.enqueued = 0;
    }

    /// A whole epoch's steps in one call (device model): the improving steps in order, each with its eval — what the
    /// example prints and logs per step (04-c21-tree.rs:144-148) — and the final `ArgminData` refreshed.
    pub fn par_roll_out_epoch(&mut self, episodes: u32, n_as_tol: impl Fn(usize) -> u32 + Sync) -> Vec<(u32, f32)> {
        assert!(self.model.is_none(), "par_roll_out_epoch needs the device model");
        self.check_tol(&n_as_tol);
        let mut log = vec![sys::azb_improvement::default(); episodes as usize];
        let mut n: u32 = 0;
        ck(self.h, unsafe { sys::azb_step(self.h, episodes, log.as_mut_ptr(), episodes, &mut n) });
        if n > 0 {
            self.refresh_argmin(true);
        }
        log.truncate((n as usize).min(episodes as usize));
        log.iter().map(|r| (r.step, r.eval)).collect()
    }

    pub fn argmin_data(&self) -> &ArgminData<State<N>, Cost> {
        &self.argmin_data
    }

    /// The `k` best isomorphism classes among every node the trees hold (azb_best_trees, an extension with no
    /// reference item), ascending by (eval, canonical code).  Call it before `par_reset_trees`, which discards the trees.
    pub fn best_trees(&mut self, k: u32) -> Vec<BestTree<N>> {
        if self.enqueued > 0 {
            self.finish_batch();
        }
        let kk = k.max(1) as usize;
        let (mut eval, mut codes, mut tree, mut node) = (vec![0f32; kk], vec![0u64; 2 * kk], vec![0u32; kk], vec![0u32; kk]);
        let (mut parents, mut mask, mut l1, mut mu) = (vec![0u8; kk * N], vec![0u32; kk * Self::W], vec![0f64; kk], vec![0u32; kk]);
        let mut n: u32 = 0;
        ck(self.h, unsafe {
            sys::azb_best_trees(self.h, k, &mut n, eval.as_mut_ptr(), codes.as_mut_ptr(), tree.as_mut_ptr(), node.as_mut_ptr(),
                                parents.as_mut_ptr(), mask.as_mut_ptr(), l1.as_mut_ptr(), mu.as_mut_ptr())
        });
        (0..n as usize)
            .map(|i| BestTree {
                eval: eval[i],
                lambda_1: l1[i],
                mu: mu[i],
                state: unflatten::<N>(&parents[i * N..(i + 1) * N], &mask[i * Self::W..(i + 1) * Self::W]),
                code: [codes[2 * i], codes[2 * i + 1]],
                tree: tree[i],
                node: node[i],
            })
            .collect()
    }

    /// `par_update_model` (optimizer/mod.rs:249-281).  Device model: observations, f32 forward/backward and the Adam
    /// step never leave the GPU (all-reduced over NCCL when a communicator is attached).  Host model: the library
    /// writes root vectors, observations and weights (tree/mod.rs:242-264), the model trains on the host.
    pub fn par_update_model(&mut self, n_obs_tol: u32) -> f32 {
        if self.enqueued > 0 {
            self.finish_batch();
        }
        if let Some(m) = self.model.as_mut() {
            ck(self.h, unsafe {
                sys::azb_write_observations(self.h, n_obs_tol, self.state_vecs.as_mut_ptr(), self.h_theta_host.as_mut_ptr(), self.action_weights.as_mut_ptr())
            });
            m.update_model(&self.state_vecs, &self.h_theta_host, &self.action_weights)
        } else {
            let mut loss = 0f32;
            ck(self.h, unsafe { sys::azb_update_model(self.h, n_obs_tol, &mut loss) });
            loss
        }
    }

    /// `node_data()` of one tree (tree/mod.rs:302-307): (path, weight) pairs in `BTreeMap<ActionSet, _>` order — the
    /// empty set, i.e. the root, first (04-c21-tree.rs:174 relies on it).
    pub fn node_data(&self, tree: usize) -> Vec<(ActionSet, NodeWeight)> {
        let (mut nn, mut na, mut np) = (0u32, 0u32, 0u32);
        ck(self.h, unsafe { sys::azb_tree_sizes(self.h, tree as u32, &mut nn, &mut na, &mut np) });
        let mut nodes = vec![0u32; nn as usize * 6];
        let mut keys = vec![0u32; nn as usize * Self::W];
        let mut preds = vec![0u32; np as usize * 3];
        let mut arcs = vec![0u32; na as usize * 3];
        ck(self.h, unsafe { sys::azb_dump_tree(self.h, tree as u32, nodes.as_mut_ptr(), keys.as_mut_ptr(), preds.as_mut_ptr(), arcs.as_mut_ptr()) });
        let mut out: Vec<(ActionSet, NodeWeight)> = (0..nn as usize)
            .map(|i| {
                let mut p = ActionSet::new();
                for a in 0..Self::A {
                    if keys[i * Self::W + a / 32] >> (a % 32) & 1 == 1 {
                        unsafe { p.push_unchecked(a) };
                    }
                }
                (p, NodeWeight { c: f32::from_bits(nodes[i * 6]), c_star: f32::from_bits(nodes[i * 6 + 1]) })
            })
            .collect();
        out.sort_by(|a, b| a.0.cmp(&b.0));
        out
    }

    /// `par_reset_trees` (optimizer/mod.rs:284-360) with an arbitrary `modify_root` closure, evaluated on the host
    /// over `node_data()` exactly like the reference; the new roots are uploaded and the trees re-seeded.
    pub fn par_reset_trees(&mut self, modify_root: impl Fn(&Space<N>, &mut State<N>, Vec<(&ActionSet, &NodeWeight)>)) {
        if self.enqueued > 0 {
            self.finish_batch();
        }
        for t in 0..self.batch {
            let data = self.node_data(t);
            let view: Vec<(&ActionSet, &NodeWeight)> = data.iter().map(|(p, w)| (p, w)).collect();
            modify_root(&self.space, &mut self.roots[t], view);
        }
        self.upload_roots_and_init();
    }

    /// The same with the example's policy (04-c21-tree.rs:172-206) evaluated on the device: no tree leaves the GPU.
    /// Draws come from a counter hash of (seed, reset count, global root index) instead of `thread_rng`.
    pub fn par_reset_trees_c21(&mut self, k_min: u32, k_max: u32) {
        if self.enqueued > 0 {
            self.finish_batch();
        }
        self.reset_seed = self.reset_seed.wrapping_mul(0x9E37_79B9_7F4A_7C15).wrapping_add(1);
        ck(self.h, unsafe { sys::azb_reset_trees(self.h, self.reset_seed, k_min, k_max) });
        let mut parents = vec![0u8; self.batch * N];
        let mut masks = vec![0u32; self.batch * Self::W];
        ck(self.h, unsafe { sys::azb_get_roots(self.h, parents.as_mut_ptr(), masks.as_mut_ptr()) });
        for (i, r) in self.roots.iter_mut().enumerate() {
            *r = unflatten::<N>(&parents[i * N..(i + 1) * N], &masks[i * Self::W..(i + 1) * Self::W]);
        }
    }

    /// Sharded runs: attach the NCCL communicator used only at the epoch boundary (include/azb.h).
    pub fn comm_init(&mut self, id128: &[u8; 128], rank: i32, world: i32) {
        ck(self.h, unsafe { sys::azb_comm_init(self.h, id128.as_ptr(), rank, world) });
    }

    /// The global `ArgminData` over every rank's roots and the rank that owns it.
    pub fn comm_argmin(&mut self) -> (ArgminData<State<N>, Cost>, i32) {
        let mut parents = vec![0u8; N];
        let mut mask = vec![0u32; Self::W];
        let (mut l1, mut mu, mut eval, mut owner) = (0f64, 0u32, 0f32, 0 as c_int);
        ck(self.h, unsafe {
            sys::azb_comm_argmin(self.h, parents.as_mut_ptr(), mask.as_mut_ptr(), &mut l1, &mut mu, &mut eval, &mut owner)
        });
        let state = unflatten::<N>(&parents, &mask);
        let cost = cost_of::<N>(&state, l1, mu, true);
        (ArgminData::new(state, cost, eval), owner)
    }
}

impl<const N: usize, M> Drop for B200Optimizer<N, M> {
    fn drop(&mut self) {
        unsafe { sys::azb_destroy(self.h) };
    }
}
