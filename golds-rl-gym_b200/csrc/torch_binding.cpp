// libswarm_b200_torch.so -- the C ABI of include/swarm_b200.h exposed as a PyTorch extension:
//   torch.ops.swarm_b200.{step, step_final, step_host, reset, rasterize, expand_obs, clip_actions, forces,
//                         reset_physics, step_physics, forces_physics}
// Each op checks device / dtype / contiguity / shape of its tensors, takes the CURRENT CUDA stream of
// the tensors' device and forwards plain pointers to the extern "C" entry point of libswarm_b200.so.
// No arithmetic happens here.  `params` is a CPU uint8 tensor holding the SwarmParams POD
// (ctypes struct bytes), so that the op signatures stay short and the struct has one definition.
#include <ATen/ATen.h>
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/library.h>

#include <cstring>

#include "../../include/swarm_b200.h"

namespace {

SwarmParams unpack(const at::Tensor& params) {
    TORCH_CHECK(params.device().is_cpu() && params.scalar_type() == at::kByte && params.is_contiguous() &&
                    params.numel() == (int64_t)sizeof(SwarmParams),
                "params must be a contiguous CPU uint8 tensor of sizeof(SwarmParams) = ", sizeof(SwarmParams), " bytes");
    SwarmParams p;
    std::memcpy(&p, params.data_ptr(), sizeof(p));
    return p;
}

void need(const at::Tensor& t, at::ScalarType dt, std::initializer_list<int64_t> shape, const char* name) {
    TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor");
    TORCH_CHECK(t.scalar_type() == dt, name, " has dtype ", t.scalar_type(), ", expected ", dt);
    TORCH_CHECK(t.is_contiguous(), name, " must be contiguous");
    TORCH_CHECK(t.sizes() == at::IntArrayRef(shape), name, " has shape ", t.sizes(), ", expected ", at::IntArrayRef(shape));
}

void check(int rc, const char* what) {
    if (rc == SWARM_OK) return;
    if (rc == SWARM_ERR_LAUNCH) TORCH_CHECK(false, what, " failed: ", swarm_strerror(rc), ": ", swarm_last_cuda_error());
    TORCH_CHECK(false, what, " failed (", rc, "): ", swarm_strerror(rc));
}

template <typename T>
T* ptr(const c10::optional<at::Tensor>& t) { return t.has_value() ? t->data_ptr<T>() : nullptr; }

swarm_stream_t stream_of(const at::Tensor& t) { return (swarm_stream_t)c10::cuda::getCurrentCUDAStream(t.get_device()).stream(); }

SwarmState make_state(const SwarmParams& p, const at::Tensor& x, const at::Tensor& xa, const at::Tensor& noise_x,
                      const at::Tensor& noise_a, const at::Tensor& elapsed, const at::Tensor& episode,
                      const c10::optional<at::Tensor>& work = c10::nullopt) {
    const int64_t E = p.n_envs, N = p.n_locusts, A = p.n_agents;
    need(x, at::kDouble, {E, N, 2}, "x");
    need(xa, at::kDouble, {E, A, 2}, "xa");
    need(noise_x, at::kDouble, {E, N, 2}, "noise_x");
    need(noise_a, at::kDouble, {E, A, 2}, "noise_a");
    need(elapsed, at::kInt, {E}, "elapsed");
    need(episode, at::kInt, {E}, "episode");
    if (work.has_value()) {
        TORCH_CHECK(work->is_cuda() && work->scalar_type() == at::kInt && work->is_contiguous() && work->dim() == 1,
                    "work must be a contiguous 1-D int32 CUDA tensor");
        TORCH_CHECK(work->get_device() == x.get_device(), "work is on another device than x");
    }
    for (const at::Tensor* t : {&xa, &noise_x, &noise_a, &elapsed, &episode})
        TORCH_CHECK(t->get_device() == x.get_device(), "all state tensors must be on the same device");
    return SwarmState{x.data_ptr<double>(), xa.data_ptr<double>(), noise_x.data_ptr<double>(), noise_a.data_ptr<double>(),
                      elapsed.data_ptr<int32_t>(), reinterpret_cast<uint32_t*>(episode.data_ptr<int32_t>()),
                      work.has_value() ? reinterpret_cast<uint32_t*>(work->data_ptr<int32_t>()) : nullptr,
                      work.has_value() ? (uint64_t)work->numel() : 0};
}

SwarmStepIO make_io(const SwarmParams& p, const at::Tensor& actions, const c10::optional<at::Tensor>& noise_a_step,
                    const c10::optional<at::Tensor>& noise_x_step, const at::Tensor& reward, const at::Tensor& done,
                    const c10::optional<at::Tensor>& grid, const c10::optional<at::Tensor>& positions,
                    const c10::optional<at::Tensor>& v_out, int64_t flags) {
    const int64_t E = p.n_envs, N = p.n_locusts, A = p.n_agents, G = p.grid_size;
    SwarmStepIO io;
    std::memset(&io, 0, sizeof(io));
    io.flags = (uint32_t)flags & ~SWARM_STEP_ACTIONS_F64;
    if (actions.scalar_type() == at::kDouble) {
        need(actions, at::kDouble, {E, A, 2}, "actions");
        io.actions_f64 = actions.data_ptr<double>();
        io.flags |= SWARM_STEP_ACTIONS_F64;
    } else {
        need(actions, at::kFloat, {E, A, 2}, "actions");
        io.actions_f32 = actions.data_ptr<float>();
    }
    if (noise_a_step.has_value()) need(*noise_a_step, at::kDouble, {E, A, 2}, "noise_a_step");
    if (noise_x_step.has_value()) need(*noise_x_step, at::kDouble, {E, N, 2}, "noise_x_step");
    io.noise_a = ptr<double>(noise_a_step);
    io.noise_x = ptr<double>(noise_x_step);
    need(reward, at::kFloat, {E}, "reward");
    need(done, at::kByte, {E}, "done");
    io.reward = reward.data_ptr<float>();
    io.done = done.data_ptr<uint8_t>();
    if (grid.has_value()) need(*grid, at::kFloat, {E, G, G, 2}, "grid");
    if (positions.has_value()) need(*positions, at::kByte, {E, A, 2}, "positions");
    if (v_out.has_value()) need(*v_out, at::kFloat, {E, N, 2}, "v_out");
    io.grid = ptr<float>(grid);
    io.positions = ptr<uint8_t>(positions);
    io.v_out = ptr<float>(v_out);
    return io;
}

SwarmInjectedDraws make_draws(const SwarmParams& p, const at::TensorList& d) {
    TORCH_CHECK(d.size() == 5, "draws must be [x0, xa0, burn_actions, agent_noise, particle_noise]");
    const int64_t E = p.n_envs, N = p.n_locusts, A = p.n_agents, B = p.n_burn_in;
    need(d[0], at::kDouble, {E, N, 2}, "draws.x0");
    need(d[1], at::kDouble, {E, A, 2}, "draws.xa0");
    need(d[2], at::kDouble, {E, B, A, 2}, "draws.burn_actions");
    need(d[3], at::kDouble, {E, B + 1, A, 2}, "draws.agent_noise");
    need(d[4], at::kDouble, {E, B + 1, N, 2}, "draws.particle_noise");
    return SwarmInjectedDraws{d[0].data_ptr<double>(), d[1].data_ptr<double>(), d[2].data_ptr<double>(),
                              d[3].data_ptr<double>(), d[4].data_ptr<double>()};
}

// SwarmEnv._step + TimeLimit (+ auto-reset, + process_state): one kernel launch on the current stream
void op_step(const at::Tensor& params, at::Tensor x, at::Tensor xa, at::Tensor noise_x, at::Tensor noise_a, at::Tensor elapsed,
             at::Tensor episode, c10::optional<at::Tensor> work, at::Tensor actions, c10::optional<at::Tensor> noise_a_step,
             c10::optional<at::Tensor> noise_x_step, at::Tensor reward, at::Tensor done, c10::optional<at::Tensor> grid,
             c10::optional<at::Tensor> positions, c10::optional<at::Tensor> v_out, int64_t flags, at::TensorList reset_draws) {
    const SwarmParams p = unpack(params);
    c10::cuda::CUDAGuard guard(x.device());
    const SwarmState st = make_state(p, x, xa, noise_x, noise_a, elapsed, episode, work);
    const SwarmStepIO io = make_io(p, actions, noise_a_step, noise_x_step, reward, done, grid, positions, v_out, flags);
    TORCH_CHECK(actions.get_device() == x.get_device() && reward.get_device() == x.get_device() &&
                    done.get_device() == x.get_device() && (!grid.has_value() || grid->get_device() == x.get_device()) &&
                    (!positions.has_value() || positions->get_device() == x.get_device()),
                "step: all tensors must be on x's device");
    SwarmInjectedDraws dr;
    if (reset_draws.size()) dr = make_draws(p, reset_draws);
    check(swarm_step(&p, &st, &io, reset_draws.size() ? &dr : nullptr, stream_of(x)), "swarm_step");
}

// op_step + what the auto-reset overwrites (swarm_step_final): the done split, the terminal state and, with final_grid,
// the terminal observation of the envs that are done
void op_step_final(const at::Tensor& params, at::Tensor x, at::Tensor xa, at::Tensor noise_x, at::Tensor noise_a,
                   at::Tensor elapsed, at::Tensor episode, c10::optional<at::Tensor> work, at::Tensor actions,
                   c10::optional<at::Tensor> noise_a_step, c10::optional<at::Tensor> noise_x_step, at::Tensor reward,
                   at::Tensor done, c10::optional<at::Tensor> grid, c10::optional<at::Tensor> positions,
                   c10::optional<at::Tensor> v_out, int64_t flags, at::TensorList reset_draws,
                   c10::optional<at::Tensor> final_x, c10::optional<at::Tensor> final_xa,
                   c10::optional<at::Tensor> terminated, c10::optional<at::Tensor> truncated,
                   c10::optional<at::Tensor> final_grid, c10::optional<at::Tensor> final_positions) {
    const SwarmParams p = unpack(params);
    c10::cuda::CUDAGuard guard(x.device());
    const SwarmState st = make_state(p, x, xa, noise_x, noise_a, elapsed, episode, work);
    const SwarmStepIO io = make_io(p, actions, noise_a_step, noise_x_step, reward, done, grid, positions, v_out, flags);
    const int64_t E = p.n_envs, N = p.n_locusts, A = p.n_agents, G = p.grid_size;
    if (final_x.has_value()) need(*final_x, at::kDouble, {E, N, 2}, "final_x");
    if (final_xa.has_value()) need(*final_xa, at::kDouble, {E, A, 2}, "final_xa");
    if (terminated.has_value()) need(*terminated, at::kByte, {E}, "terminated");
    if (truncated.has_value()) need(*truncated, at::kByte, {E}, "truncated");
    if (final_grid.has_value()) need(*final_grid, at::kFloat, {E, G, G, 2}, "final_grid");
    if (final_positions.has_value()) need(*final_positions, at::kByte, {E, A, 2}, "final_positions");
    bool same = actions.get_device() == x.get_device() && reward.get_device() == x.get_device() &&
                done.get_device() == x.get_device();
    for (const c10::optional<at::Tensor>* t : {&grid, &positions, &final_x, &final_xa, &terminated, &truncated, &final_grid,
                                               &final_positions})
        same = same && (!t->has_value() || (*t)->get_device() == x.get_device());
    TORCH_CHECK(same, "step_final: all tensors must be on x's device");
    SwarmInjectedDraws dr;
    if (reset_draws.size()) dr = make_draws(p, reset_draws);
    const SwarmStepFinal fin{ptr<double>(final_x), ptr<double>(final_xa), ptr<uint8_t>(terminated), ptr<uint8_t>(truncated),
                             ptr<float>(final_grid), ptr<uint8_t>(final_positions)};
    check(swarm_step_final(&p, &st, &io, &fin, reset_draws.size() ? &dr : nullptr, stream_of(x)), "swarm_step_final");
}

// SwarmPhysics of the *_physics ops: the (E,6) f64 table on x's device, the flags and the per-column ranges
SwarmPhysics make_physics(const SwarmParams& p, const at::Tensor& table, int64_t flags, at::ArrayRef<double> lo,
                          at::ArrayRef<double> hi, const at::Tensor& x) {
    need(table, at::kDouble, {p.n_envs, 6}, "physics");
    TORCH_CHECK(table.get_device() == x.get_device(), "physics is on another device than x");
    TORCH_CHECK(lo.size() == 6 && hi.size() == 6, "physics_lo and physics_hi must have 6 entries");
    SwarmPhysics ph;
    std::memset(&ph, 0, sizeof(ph));
    ph.table = table.data_ptr<double>();
    ph.flags = (uint32_t)flags;
    for (int c = 0; c < 6; ++c) {
        ph.lo[c] = lo[c];
        ph.hi[c] = hi[c];
    }
    return ph;
}

void op_reset(const at::Tensor& params, at::Tensor x, at::Tensor xa, at::Tensor noise_x, at::Tensor noise_a, at::Tensor elapsed,
              at::Tensor episode, c10::optional<at::Tensor> mask, at::TensorList draws) {
    const SwarmParams p = unpack(params);
    c10::cuda::CUDAGuard guard(x.device());
    const SwarmState st = make_state(p, x, xa, noise_x, noise_a, elapsed, episode);
    if (mask.has_value()) need(*mask, at::kByte, {p.n_envs}, "mask");
    SwarmInjectedDraws dr;
    if (draws.size()) dr = make_draws(p, draws);
    check(swarm_reset(&p, &st, ptr<uint8_t>(mask), draws.size() ? &dr : nullptr, stream_of(x)), "swarm_reset");
}

void op_rasterize(const at::Tensor& params, const at::Tensor& x, const c10::optional<at::Tensor>& xa, at::Tensor grid,
                  c10::optional<at::Tensor> positions, c10::optional<at::Tensor> box) {
    const SwarmParams p = unpack(params);
    c10::cuda::CUDAGuard guard(x.device());
    const int64_t E = p.n_envs, N = p.n_locusts, A = p.n_agents, G = p.grid_size;
    need(x, at::kDouble, {E, N, 2}, "x");
    if (A > 0) {
        TORCH_CHECK(xa.has_value() && positions.has_value(), "xa and positions are required when n_agents > 0");
        need(*xa, at::kDouble, {E, A, 2}, "xa");
        need(*positions, at::kByte, {E, A, 2}, "positions");
    }
    need(grid, at::kFloat, {E, G, G, 2}, "grid");
    if (box.has_value()) need(*box, at::kDouble, {E, 4}, "box");
    check(swarm_rasterize(&p, x.data_ptr<double>(), A > 0 ? xa->data_ptr<double>() : nullptr, grid.data_ptr<float>(),
                          A > 0 ? positions->data_ptr<uint8_t>() : nullptr, ptr<double>(box), stream_of(x)),
          "swarm_rasterize");
}

void op_expand_obs(const at::Tensor& params, const at::Tensor& grid, const at::Tensor& positions, at::Tensor expanded) {
    const SwarmParams p = unpack(params);
    c10::cuda::CUDAGuard guard(grid.device());
    const int64_t E = p.n_envs, A = p.n_agents, G = p.grid_size;
    need(grid, at::kFloat, {E, G, G, 2}, "grid");
    need(positions, at::kByte, {E, A, 2}, "positions");
    need(expanded, at::kFloat, {E, A, G, G, 3}, "expanded");
    check(swarm_expand_obs(&p, grid.data_ptr<float>(), positions.data_ptr<uint8_t>(), expanded.data_ptr<float>(),
                           stream_of(grid)), "swarm_expand_obs");
}

void op_clip_actions(at::Tensor actions, double max_norm) {
    TORCH_CHECK(actions.is_cuda() && actions.scalar_type() == at::kFloat && actions.is_contiguous() &&
                    actions.dim() >= 1 && actions.size(-1) == 2,
                "actions must be a contiguous float32 (...,2) CUDA tensor");
    c10::cuda::CUDAGuard guard(actions.device());
    check(swarm_clip_actions(actions.data_ptr<float>(), actions.numel() / 2, (float)max_norm, stream_of(actions)),
          "swarm_clip_actions");
}

void op_forces(const at::Tensor& params, const at::Tensor& x, const at::Tensor& xa, c10::optional<at::Tensor> v,
               c10::optional<at::Tensor> reward) {
    const SwarmParams p = unpack(params);
    c10::cuda::CUDAGuard guard(x.device());
    const int64_t E = p.n_envs, N = p.n_locusts, A = p.n_agents;
    need(x, at::kDouble, {E, N, 2}, "x");
    need(xa, at::kDouble, {E, A, 2}, "xa");
    if (v.has_value()) need(*v, at::kFloat, {E, N, 2}, "v");
    if (reward.has_value()) need(*reward, at::kFloat, {E}, "reward");
    check(swarm_forces(&p, x.data_ptr<double>(), xa.data_ptr<double>(), ptr<float>(v), ptr<float>(reward), stream_of(x)),
          "swarm_forces");
}

void op_reset_physics(const at::Tensor& params, at::Tensor x, at::Tensor xa, at::Tensor noise_x, at::Tensor noise_a,
                      at::Tensor elapsed, at::Tensor episode, c10::optional<at::Tensor> mask, at::TensorList draws,
                      at::Tensor physics, int64_t physics_flags, at::ArrayRef<double> physics_lo,
                      at::ArrayRef<double> physics_hi) {
    const SwarmParams p = unpack(params);
    c10::cuda::CUDAGuard guard(x.device());
    const SwarmState st = make_state(p, x, xa, noise_x, noise_a, elapsed, episode);
    if (mask.has_value()) need(*mask, at::kByte, {p.n_envs}, "mask");
    SwarmInjectedDraws dr;
    if (draws.size()) dr = make_draws(p, draws);
    const SwarmPhysics ph = make_physics(p, physics, physics_flags, physics_lo, physics_hi, x);
    check(swarm_reset_physics(&p, &st, &ph, ptr<uint8_t>(mask), draws.size() ? &dr : nullptr, stream_of(x)),
          "swarm_reset_physics");
}

// op_step_final with per-env physics; without any of the final_* / terminated / truncated tensors it is op_step's call
void op_step_physics(const at::Tensor& params, at::Tensor x, at::Tensor xa, at::Tensor noise_x, at::Tensor noise_a,
                     at::Tensor elapsed, at::Tensor episode, c10::optional<at::Tensor> work, at::Tensor actions,
                     c10::optional<at::Tensor> noise_a_step, c10::optional<at::Tensor> noise_x_step, at::Tensor reward,
                     at::Tensor done, c10::optional<at::Tensor> grid, c10::optional<at::Tensor> positions,
                     c10::optional<at::Tensor> v_out, int64_t flags, at::TensorList reset_draws, at::Tensor physics,
                     int64_t physics_flags, at::ArrayRef<double> physics_lo, at::ArrayRef<double> physics_hi,
                     c10::optional<at::Tensor> final_x, c10::optional<at::Tensor> final_xa,
                     c10::optional<at::Tensor> terminated, c10::optional<at::Tensor> truncated,
                     c10::optional<at::Tensor> final_grid, c10::optional<at::Tensor> final_positions) {
    const SwarmParams p = unpack(params);
    c10::cuda::CUDAGuard guard(x.device());
    const SwarmState st = make_state(p, x, xa, noise_x, noise_a, elapsed, episode, work);
    const SwarmStepIO io = make_io(p, actions, noise_a_step, noise_x_step, reward, done, grid, positions, v_out, flags);
    const int64_t E = p.n_envs, N = p.n_locusts, A = p.n_agents, G = p.grid_size;
    if (final_x.has_value()) need(*final_x, at::kDouble, {E, N, 2}, "final_x");
    if (final_xa.has_value()) need(*final_xa, at::kDouble, {E, A, 2}, "final_xa");
    if (terminated.has_value()) need(*terminated, at::kByte, {E}, "terminated");
    if (truncated.has_value()) need(*truncated, at::kByte, {E}, "truncated");
    if (final_grid.has_value()) need(*final_grid, at::kFloat, {E, G, G, 2}, "final_grid");
    if (final_positions.has_value()) need(*final_positions, at::kByte, {E, A, 2}, "final_positions");
    bool same = actions.get_device() == x.get_device() && reward.get_device() == x.get_device() &&
                done.get_device() == x.get_device();
    for (const c10::optional<at::Tensor>* t : {&grid, &positions, &final_x, &final_xa, &terminated, &truncated, &final_grid,
                                               &final_positions})
        same = same && (!t->has_value() || (*t)->get_device() == x.get_device());
    TORCH_CHECK(same, "step_physics: all tensors must be on x's device");
    const SwarmPhysics ph = make_physics(p, physics, physics_flags, physics_lo, physics_hi, x);
    SwarmInjectedDraws dr;
    if (reset_draws.size()) dr = make_draws(p, reset_draws);
    const bool any_fin = final_x.has_value() || final_xa.has_value() || terminated.has_value() || truncated.has_value() ||
                         final_grid.has_value() || final_positions.has_value();
    const SwarmStepFinal fin{ptr<double>(final_x), ptr<double>(final_xa), ptr<uint8_t>(terminated), ptr<uint8_t>(truncated),
                             ptr<float>(final_grid), ptr<uint8_t>(final_positions)};
    check(swarm_step_physics(&p, &st, &io, any_fin ? &fin : nullptr, &ph, reset_draws.size() ? &dr : nullptr, stream_of(x)),
          "swarm_step_physics");
}

void op_forces_physics(const at::Tensor& params, const at::Tensor& x, const at::Tensor& xa, c10::optional<at::Tensor> v,
                       c10::optional<at::Tensor> reward, at::Tensor physics, int64_t physics_flags,
                       at::ArrayRef<double> physics_lo, at::ArrayRef<double> physics_hi) {
    const SwarmParams p = unpack(params);
    c10::cuda::CUDAGuard guard(x.device());
    const int64_t E = p.n_envs, N = p.n_locusts, A = p.n_agents;
    need(x, at::kDouble, {E, N, 2}, "x");
    need(xa, at::kDouble, {E, A, 2}, "xa");
    if (v.has_value()) need(*v, at::kFloat, {E, N, 2}, "v");
    if (reward.has_value()) need(*reward, at::kFloat, {E}, "reward");
    const SwarmPhysics ph = make_physics(p, physics, physics_flags, physics_lo, physics_hi, x);
    check(swarm_forces_physics(&p, &ph, x.data_ptr<double>(), xa.data_ptr<double>(), ptr<float>(v), ptr<float>(reward),
                               stream_of(x)),
          "swarm_forces_physics");
}

int64_t op_abi_version() { return swarm_abi_version(); }

}  // namespace

TORCH_LIBRARY(swarm_b200, m) {
    m.def("step(Tensor params, Tensor(a!) x, Tensor(b!) xa, Tensor(c!) noise_x, Tensor(d!) noise_a, Tensor(e!) elapsed, "
          "Tensor(f!) episode, Tensor(m!)? work, Tensor(g!) actions, Tensor? noise_a_step, Tensor? noise_x_step, Tensor(h!) reward, "
          "Tensor(i!) done, Tensor(j!)? grid, Tensor(k!)? positions, Tensor(l!)? v_out, int flags, Tensor[] reset_draws) -> ()",
          &op_step);
    m.def("step_final(Tensor params, Tensor(a!) x, Tensor(b!) xa, Tensor(c!) noise_x, Tensor(d!) noise_a, Tensor(e!) elapsed, "
          "Tensor(f!) episode, Tensor(m!)? work, Tensor(g!) actions, Tensor? noise_a_step, Tensor? noise_x_step, "
          "Tensor(h!) reward, Tensor(i!) done, Tensor(j!)? grid, Tensor(k!)? positions, Tensor(l!)? v_out, int flags, "
          "Tensor[] reset_draws, Tensor(n!)? final_x, Tensor(o!)? final_xa, Tensor(p!)? terminated, Tensor(q!)? truncated, "
          "Tensor(r!)? final_grid, Tensor(s!)? final_positions) -> ()",
          &op_step_final);
    m.def("reset(Tensor params, Tensor(a!) x, Tensor(b!) xa, Tensor(c!) noise_x, Tensor(d!) noise_a, Tensor(e!) elapsed, "
          "Tensor(f!) episode, Tensor? mask, Tensor[] draws) -> ()", &op_reset);
    m.def("rasterize(Tensor params, Tensor x, Tensor? xa, Tensor(a!) grid, Tensor(b!)? positions, Tensor(c!)? box) -> ()",
          &op_rasterize);
    m.def("expand_obs(Tensor params, Tensor grid, Tensor positions, Tensor(a!) expanded) -> ()", &op_expand_obs);
    m.def("clip_actions(Tensor(a!) actions, float max_norm) -> ()", &op_clip_actions);
    m.def("forces(Tensor params, Tensor x, Tensor xa, Tensor(a!)? v, Tensor(b!)? reward) -> ()", &op_forces);
    m.def("reset_physics(Tensor params, Tensor(a!) x, Tensor(b!) xa, Tensor(c!) noise_x, Tensor(d!) noise_a, "
          "Tensor(e!) elapsed, Tensor(f!) episode, Tensor? mask, Tensor[] draws, Tensor(g!) physics, int physics_flags, "
          "float[] physics_lo, float[] physics_hi) -> ()", &op_reset_physics);
    m.def("step_physics(Tensor params, Tensor(a!) x, Tensor(b!) xa, Tensor(c!) noise_x, Tensor(d!) noise_a, "
          "Tensor(e!) elapsed, Tensor(f!) episode, Tensor(m!)? work, Tensor(g!) actions, Tensor? noise_a_step, "
          "Tensor? noise_x_step, Tensor(h!) reward, Tensor(i!) done, Tensor(j!)? grid, Tensor(k!)? positions, "
          "Tensor(l!)? v_out, int flags, Tensor[] reset_draws, Tensor(t!) physics, int physics_flags, float[] physics_lo, "
          "float[] physics_hi, Tensor(n!)? final_x, Tensor(o!)? final_xa, Tensor(p!)? terminated, Tensor(q!)? truncated, "
          "Tensor(r!)? final_grid, Tensor(s!)? final_positions) -> ()",
          &op_step_physics);
    m.def("forces_physics(Tensor params, Tensor x, Tensor xa, Tensor(a!)? v, Tensor(b!)? reward, Tensor physics, "
          "int physics_flags, float[] physics_lo, float[] physics_hi) -> ()", &op_forces_physics);
    m.def("abi_version() -> int", &op_abi_version);
}
