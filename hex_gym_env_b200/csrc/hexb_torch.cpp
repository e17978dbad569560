// hexb_torch.cpp - the C ABI of include/hexb.h exposed as PyTorch operators (torch.ops.hexb.*).
//
// BASELINE north star: "Python host code calling the hot path through a thin C-ABI layer exposed as a PyTorch extension".
// This file is that layer and nothing more: every operator validates its tensors (device, dtype, contiguity, element count
// against the handle's configuration), takes the CURRENT CUDA stream of the handle's device, and forwards raw device pointers
// to the corresponding extern "C" entry point of libhexb.so. No kernel, no game logic and no CPU path live here. Operators
// that write tensors declare them mutable (Tensor(a!)), so they are usable under torch's functionalisation / CUDA-graph capture.
//
// The environment handle (hexb_env*) travels as an int64, exactly like the ctypes binding passes it (hex_gym_env_b200/_native.py).
// Build: hex_gym_env_b200/torch_ops.py (g++ against the torch headers, linked to libhexb.so with rpath $ORIGIN).
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/library.h>

#include "../include/hexb.h"

namespace {

using at::Tensor;
using OptT = const std::optional<Tensor> &;

hexb_env *env_of(int64_t handle) {
    TORCH_CHECK(handle != 0, "hexb: null environment handle");
    return reinterpret_cast<hexb_env *>(static_cast<intptr_t>(handle));
}

hexb_config config_of(hexb_env *e) {
    hexb_config c;
    TORCH_CHECK(hexb_get_config(e, &c) == HEXB_OK, "hexb: bad environment handle");
    return c;
}

void check_rc(int32_t rc, const char *what) {
    if (rc == HEXB_OK) return;
    if (rc == HEXB_ERR_CUDA) TORCH_CHECK(false, "hexb::", what, ": ", hexb_strerror(rc), " (cudaError ", hexb_last_cuda_error(), ")");
    TORCH_CHECK(false, "hexb::", what, ": ", hexb_strerror(rc));
}

// raw pointer of an optional tensor after checking that it is what the C ABI expects
template <class T>
T *ptr(OptT t, c10::ScalarType dtype, int64_t numel, int device, const char *name) {
    if (!t.has_value() || !t->defined()) return nullptr;
    TORCH_CHECK(t->is_cuda() && t->get_device() == device, "hexb: ", name, " must live on cuda:", device);
    TORCH_CHECK(t->scalar_type() == dtype, "hexb: ", name, " must have dtype ", c10::toString(dtype));
    TORCH_CHECK(t->is_contiguous(), "hexb: ", name, " must be contiguous");
    TORCH_CHECK(t->numel() == numel, "hexb: ", name, " must have ", numel, " elements, got ", t->numel());
    return reinterpret_cast<T *>(t->data_ptr());
}

struct Call {
    hexb_env *e;
    hexb_config c;
    int64_t G, C;
    c10::cuda::CUDAGuard guard;
    void *stream;
    c10::ScalarType obs_t() const { return c.obs_dtype == HEXB_OBS_F32 ? at::kFloat : at::kChar; }   // hexb_config.obs_dtype
    explicit Call(int64_t handle) : e(env_of(handle)), c(config_of(e)), G(c.num_games), C((int64_t)c.board_size * c.board_size), guard(c.device) {
        stream = at::cuda::getCurrentCUDAStream(c.device).stream();
    }
};

void op_reset(int64_t handle, OptT reset_mask, OptT open_u, OptT obs, OptT mask) {
    Call k(handle);
    const int d = k.c.device;
    check_rc(hexb_reset(k.e, ptr<const uint8_t>(reset_mask, at::kByte, k.G, d, "reset_mask"), ptr<const double>(open_u, at::kDouble, k.G, d, "open_u"),
                        ptr<void>(obs, k.obs_t(), k.G * k.C, d, "obs"), ptr<uint8_t>(mask, at::kByte, k.G * k.C, d, "mask"), k.stream),
             "reset");
}

void op_step(int64_t handle, OptT actions, OptT opp_u, OptT obs, OptT mask, OptT reward, OptT done, OptT term_obs, OptT actions_out) {
    Call k(handle);
    const int d = k.c.device;
    check_rc(hexb_step(k.e, ptr<const int32_t>(actions, at::kInt, k.G, d, "actions"), ptr<const double>(opp_u, at::kDouble, 2 * k.G, d, "opp_u"),
                       ptr<void>(obs, k.obs_t(), k.G * k.C, d, "obs"), ptr<uint8_t>(mask, at::kByte, k.G * k.C, d, "mask"),
                       ptr<float>(reward, at::kFloat, k.G, d, "reward"), ptr<uint8_t>(done, at::kByte, k.G, d, "done"),
                       ptr<void>(term_obs, k.obs_t(), k.G * k.C, d, "term_obs"), ptr<int32_t>(actions_out, at::kInt, k.G, d, "actions_out"),
                       k.stream),
             "step");
}

void op_rollout(int64_t handle, int64_t num_steps, OptT obs, OptT mask, OptT reward, OptT done, OptT term_obs, OptT actions_out) {
    Call k(handle);
    const int d = k.c.device;
    TORCH_CHECK(num_steps >= 1 && num_steps <= 65536, "hexb::rollout: num_steps out of range");
    const int64_t T = num_steps;
    check_rc(hexb_rollout(k.e, (int32_t)T, ptr<void>(obs, k.obs_t(), T * k.G * k.C, d, "obs"), ptr<uint8_t>(mask, at::kByte, T * k.G * k.C, d, "mask"),
                          ptr<float>(reward, at::kFloat, T * k.G, d, "reward"), ptr<uint8_t>(done, at::kByte, T * k.G, d, "done"),
                          ptr<void>(term_obs, k.obs_t(), T * k.G * k.C, d, "term_obs"),
                          ptr<int32_t>(actions_out, at::kInt, T * k.G, d, "actions_out"), k.stream),
             "rollout");
}

void op_half_step(int64_t handle, int64_t side, OptT actions, OptT reward, OptT done, OptT term_obs) {
    Call k(handle);
    const int d = k.c.device;
    check_rc(hexb_half_step(k.e, (int32_t)side, ptr<const int32_t>(actions, at::kInt, k.G, d, "actions"), ptr<float>(reward, at::kFloat, k.G, d, "reward"),
                            ptr<uint8_t>(done, at::kByte, k.G, d, "done"), ptr<void>(term_obs, k.obs_t(), k.G * k.C, d, "term_obs"), k.stream),
             "half_step");
}

void op_ply(int64_t handle, const Tensor &actions, OptT ret) {
    Call k(handle);
    const int d = k.c.device;
    check_rc(hexb_ply(k.e, ptr<const int32_t>(actions, at::kInt, k.G, d, "actions"), ptr<int8_t>(ret, at::kChar, k.G, d, "ret"), k.stream), "ply");
}

void op_encode(int64_t handle, int64_t view, OptT obs, OptT mask) {
    Call k(handle);
    const int d = k.c.device;
    check_rc(hexb_encode(k.e, (int32_t)view, ptr<void>(obs, k.obs_t(), k.G * k.C, d, "obs"), ptr<uint8_t>(mask, at::kByte, k.G * k.C, d, "mask"), k.stream),
             "encode");
}

void op_sample_actions(int64_t handle, int64_t view, const Tensor &u, Tensor actions_out) {
    Call k(handle);
    const int d = k.c.device;
    check_rc(hexb_sample_actions(k.e, (int32_t)view, ptr<const double>(u, at::kDouble, k.G, d, "u"), ptr<int32_t>(actions_out, at::kInt, k.G, d, "actions_out"),
                                 k.stream),
             "sample_actions");
}

void op_stats(int64_t handle, Tensor out8) {
    Call k(handle);
    check_rc(hexb_stats(k.e, ptr<int64_t>(out8, at::kLong, 8, k.c.device, "out8"), k.stream), "stats");
}

void op_masked_sample(const Tensor &logits, const Tensor &mask, const Tensor &u, OptT actions, OptT logp, OptT entropy) {
    TORCH_CHECK(logits.is_cuda() && logits.dim() == 2, "hexb::masked_sample: logits must be a CUDA tensor [G,C]");
    const int d = logits.get_device();
    const int64_t G = logits.size(0), C = logits.size(1);
    c10::cuda::CUDAGuard guard(d);
    check_rc(hexb_masked_sample(ptr<const float>(logits, at::kFloat, G * C, d, "logits"), ptr<const uint8_t>(mask, at::kByte, G * C, d, "mask"),
                                ptr<const double>(u, at::kDouble, G, d, "u"), G, (int32_t)C, ptr<int32_t>(actions, at::kInt, G, d, "actions"),
                                ptr<float>(logp, at::kFloat, G, d, "logp"), ptr<float>(entropy, at::kFloat, G, d, "entropy"), d,
                                at::cuda::getCurrentCUDAStream(d).stream()),
             "masked_sample");
}

void op_gae(const Tensor &rewards, const Tensor &values, const Tensor &dones, double gamma, double gae_lambda, Tensor advantages, OptT returns) {
    TORCH_CHECK(rewards.is_cuda() && rewards.dim() == 2, "hexb::gae: rewards must be a CUDA tensor [T,G]");
    const int d = rewards.get_device();
    const int64_t T = rewards.size(0), G = rewards.size(1);
    c10::cuda::CUDAGuard guard(d);
    check_rc(hexb_gae(ptr<const float>(rewards, at::kFloat, T * G, d, "rewards"), ptr<const float>(values, at::kFloat, (T + 1) * G, d, "values"),
                      ptr<const uint8_t>(dones, at::kByte, T * G, d, "dones"), (int32_t)T, G, gamma, gae_lambda,
                      ptr<float>(advantages, at::kFloat, T * G, d, "advantages"), ptr<float>(returns, at::kFloat, T * G, d, "returns"), d,
                      at::cuda::getCurrentCUDAStream(d).stream()),
             "gae");
}

void op_set_launch_form(int64_t handle, int64_t warps_per_chunk) {
    check_rc(hexb_set_launch_form(env_of(handle), (int32_t)warps_per_chunk), "set_launch_form");
}

// SelfPlayEnv.set_eval at run time; eval_episode (int32[G], optional) becomes the handle's per-game evaluation-episode counter
void op_set_eval(int64_t handle, bool eval_state, OptT eval_episode) {
    Call k(handle);
    check_rc(hexb_set_eval(k.e, eval_state ? 1 : 0, ptr<int32_t>(eval_episode, at::kInt, k.G, k.c.device, "eval_episode"), k.stream), "set_eval");
}

// copy.deepcopy(env.simulator) into a raw handle: dst game dst_index[i] <- src game src_index[i] (int64[count], None = identity)
void op_copy_games(int64_t dst, int64_t src, OptT src_index, OptT dst_index, int64_t count) {
    Call k(dst);
    const hexb_config sc = config_of(env_of(src));
    TORCH_CHECK(k.c.raw, "hexb::copy_games: dst must be a raw handle");
    TORCH_CHECK(sc.board_size == k.c.board_size && sc.variant == k.c.variant && sc.device == k.c.device,
                "hexb::copy_games: src and dst differ in board_size, variant or device");
    TORCH_CHECK(count >= 0, "hexb::copy_games: count must be >= 0");
    const int d = k.c.device;
    check_rc(hexb_copy_games(k.e, env_of(src), ptr<const int64_t>(src_index, at::kLong, count, d, "src_index"),
                             ptr<const int64_t>(dst_index, at::kLong, count, d, "dst_index"), count, k.stream),
             "copy_games");
}

void op_playouts(int64_t handle, int64_t num_playouts, int64_t first_playout, OptT game_mask, Tensor wins) {
    Call k(handle);
    const int d = k.c.device;
    TORCH_CHECK(num_playouts >= 1 && num_playouts <= INT32_MAX && first_playout >= 0 && first_playout + num_playouts < (1ll << 32),
                "hexb::playouts: need num_playouts >= 1, first_playout >= 0 and first_playout + num_playouts < 2^32");
    check_rc(hexb_playouts(k.e, (int32_t)num_playouts, first_playout, ptr<const uint8_t>(game_mask, at::kByte, k.G, d, "game_mask"),
                           ptr<int32_t>(wins, at::kInt, k.G, d, "wins"), k.stream),
             "playouts");
}

// tree search (hexb_mcts_*): the tree is a uint8 tensor of at least hexb_mcts_tree_bytes bytes on the handle's device
void *tree_of(const Tensor &tree, int device) {
    TORCH_CHECK(tree.is_cuda() && tree.get_device() == device && tree.scalar_type() == at::kByte && tree.is_contiguous(),
                "hexb: tree must be a contiguous uint8 tensor on cuda:", device);
    return tree.data_ptr();
}

void op_mcts_init(int64_t handle, Tensor tree, int64_t max_nodes, double c_puct, double fpu, int64_t first_playout, OptT root_mask) {
    Call k(handle);
    const int d = k.c.device;
    TORCH_CHECK(max_nodes >= 1 && max_nodes <= INT32_MAX, "hexb::mcts_init: max_nodes out of range");
    check_rc(hexb_mcts_init(k.e, tree_of(tree, d), (size_t)tree.numel(), (int32_t)max_nodes, c_puct, fpu, first_playout,
                            ptr<const uint8_t>(root_mask, at::kByte, k.G, d, "root_mask"), k.stream),
             "mcts_init");
}

void op_mcts_search(int64_t handle, Tensor tree, int64_t num_simulations, int64_t playouts_per_leaf) {
    Call k(handle);
    TORCH_CHECK(num_simulations >= 1 && num_simulations <= INT32_MAX && playouts_per_leaf >= 1 && playouts_per_leaf <= INT32_MAX,
                "hexb::mcts_search: num_simulations and playouts_per_leaf must be >= 1");
    check_rc(hexb_mcts_search(k.e, tree_of(tree, k.c.device), (size_t)tree.numel(), (int32_t)num_simulations, (int32_t)playouts_per_leaf,
                              k.stream),
             "mcts_search");
}

void op_mcts_select(int64_t handle, Tensor tree, Tensor leaf_obs, Tensor leaf_mask, Tensor pending) {
    Call k(handle);
    const int d = k.c.device;
    check_rc(hexb_mcts_select(k.e, tree_of(tree, d), (size_t)tree.numel(), ptr<void>(leaf_obs, k.obs_t(), k.G * k.C, d, "leaf_obs"),
                              ptr<uint8_t>(leaf_mask, at::kByte, k.G * k.C, d, "leaf_mask"), ptr<uint8_t>(pending, at::kByte, k.G, d, "pending"),
                              k.stream),
             "mcts_select");
}

void op_mcts_expand(int64_t handle, Tensor tree, Tensor priors, Tensor values) {
    Call k(handle);
    const int d = k.c.device;
    check_rc(hexb_mcts_expand(k.e, tree_of(tree, d), (size_t)tree.numel(), ptr<const float>(priors, at::kFloat, k.G * k.C, d, "priors"),
                              ptr<const float>(values, at::kFloat, k.G, d, "values"), k.stream),
             "mcts_expand");
}

void op_mcts_root(int64_t handle, Tensor tree, OptT visits, OptT q, OptT value, OptT nodes_used) {
    Call k(handle);
    const int d = k.c.device;
    check_rc(hexb_mcts_root(k.e, tree_of(tree, d), (size_t)tree.numel(), ptr<int32_t>(visits, at::kInt, k.G * k.C, d, "visits"),
                            ptr<float>(q, at::kFloat, k.G * k.C, d, "q"), ptr<float>(value, at::kFloat, k.G, d, "value"),
                            ptr<int32_t>(nodes_used, at::kInt, k.G, d, "nodes_used"), k.stream),
             "mcts_root");
}

void op_mcts_advance(int64_t handle, Tensor tree, int64_t first_playout, OptT root_mask) {
    Call k(handle);
    const int d = k.c.device;
    check_rc(hexb_mcts_advance(k.e, tree_of(tree, d), (size_t)tree.numel(), first_playout,
                               ptr<const uint8_t>(root_mask, at::kByte, k.G, d, "root_mask"), k.stream),
             "mcts_advance");
}

int64_t op_version() { return hexb_version(); }

}  // namespace

TORCH_LIBRARY(hexb, m) {
    m.def("version() -> int", &op_version);
    m.def("reset(int env, Tensor? reset_mask, Tensor? open_u, Tensor(a!)? obs, Tensor(b!)? mask) -> ()");
    m.def("step(int env, Tensor? actions, Tensor? opp_u, Tensor(a!)? obs, Tensor(b!)? mask, Tensor(c!)? reward, Tensor(d!)? done, "
          "Tensor(e!)? term_obs, Tensor(f!)? actions_out) -> ()");
    m.def("rollout(int env, int num_steps, Tensor(a!)? obs, Tensor(b!)? mask, Tensor(c!)? reward, Tensor(d!)? done, Tensor(e!)? term_obs, "
          "Tensor(f!)? actions_out) -> ()");
    m.def("half_step(int env, int side, Tensor? actions, Tensor(a!)? reward, Tensor(b!)? done, Tensor(c!)? term_obs) -> ()");
    m.def("ply(int env, Tensor actions, Tensor(a!)? ret) -> ()");
    m.def("encode(int env, int view, Tensor(a!)? obs, Tensor(b!)? mask) -> ()");
    m.def("sample_actions(int env, int view, Tensor u, Tensor(a!) actions_out) -> ()");
    m.def("stats(int env, Tensor(a!) out8) -> ()");
    m.def("masked_sample(Tensor logits, Tensor mask, Tensor u, Tensor(a!)? actions, Tensor(b!)? logp, Tensor(c!)? entropy) -> ()");
    m.def("gae(Tensor rewards, Tensor values, Tensor dones, float gamma, float gae_lambda, Tensor(a!) advantages, Tensor(b!)? returns) -> ()");
    m.def("set_launch_form(int env, int warps_per_chunk) -> ()", &op_set_launch_form);
    m.def("set_eval(int env, bool eval_state, Tensor(a!)? eval_episode) -> ()");
    m.def("copy_games(int dst, int src, Tensor? src_index, Tensor? dst_index, int count) -> ()");
    m.def("playouts(int env, int num_playouts, int first_playout, Tensor? game_mask, Tensor(a!) wins) -> ()");
    m.def("mcts_init(int env, Tensor(a!) tree, int max_nodes, float c_puct, float fpu, int first_playout, Tensor? root_mask) -> ()");
    m.def("mcts_search(int env, Tensor(a!) tree, int num_simulations, int playouts_per_leaf) -> ()");
    m.def("mcts_select(int env, Tensor(a!) tree, Tensor(b!) leaf_obs, Tensor(c!) leaf_mask, Tensor(d!) pending) -> ()");
    m.def("mcts_expand(int env, Tensor(a!) tree, Tensor priors, Tensor values) -> ()");
    m.def("mcts_root(int env, Tensor tree, Tensor(a!)? visits, Tensor(b!)? q, Tensor(c!)? value, Tensor(d!)? nodes_used) -> ()");
    m.def("mcts_advance(int env, Tensor(a!) tree, int first_playout, Tensor? root_mask) -> ()");
}

// The handle is an int, so these operators have no tensor argument to dispatch on when every optional is None: register them
// for all backends (CompositeExplicitAutograd) and let the pointer checks above enforce "CUDA tensors on the handle's device".
TORCH_LIBRARY_IMPL(hexb, CompositeExplicitAutograd, m) {
    m.impl("reset", &op_reset);
    m.impl("step", &op_step);
    m.impl("rollout", &op_rollout);
    m.impl("half_step", &op_half_step);
    m.impl("ply", &op_ply);
    m.impl("encode", &op_encode);
    m.impl("sample_actions", &op_sample_actions);
    m.impl("stats", &op_stats);
    m.impl("masked_sample", &op_masked_sample);
    m.impl("gae", &op_gae);
    m.impl("set_eval", &op_set_eval);
    m.impl("copy_games", &op_copy_games);
    m.impl("playouts", &op_playouts);
    m.impl("mcts_init", &op_mcts_init);
    m.impl("mcts_search", &op_mcts_search);
    m.impl("mcts_select", &op_mcts_select);
    m.impl("mcts_expand", &op_mcts_expand);
    m.impl("mcts_root", &op_mcts_root);
    m.impl("mcts_advance", &op_mcts_advance);
}
