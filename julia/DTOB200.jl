# DTOB200.jl -- Julia glue for the B200 batched NLP-callback engine (libdto.so).
#
# Written against DirectTrajectoryOptimization.jl as vendored at /root/reference
# (Julia 1.6, Symbolics 0.1.29-0.1.32, MathOptInterface 1.3, Ipopt.jl 1.0.2; Project.toml:16-23).
# NOT EXECUTED in this repository's CI: the build image has no Julia. It is kept small and literal: every
# ccall binds one entry point of include/dto.h, the evaluator methods mirror /root/reference/src/moi.jl one
# for one, and the text it hands to the code generator is covered by fixtures that ARE tested here
# (tests/fixtures_ctarget/*.json, tests/test_frontend_cpu.py).
#
# What a user changes in a script written for the reference:
#
#     using DirectTrajectoryOptimization            # unchanged
#     using DTOB200                                 # + this module
#     dt   = DTOB200.Dynamics(f, ny, nx, nu; evaluate_hessian=true)      # same arguments as the reference's
#     ct   = DTOB200.Cost(ot, nx, nu; evaluate_hessian=true)             #   constructors (src/dynamics.jl:18,
#     con  = DTOB200.Constraint(c, nx, nu; indices_inequality=[1])       #   src/costs.jl:13, src/constraints.jl:21,
#     gen  = DTOB200.GeneralConstraint(g, nz, nw)                        #   src/general_constraint.jl:18)
#     solver = DTOB200.Solver(dynamics, objective, constraints, bounds;  # same arguments as src/solver.jl:6-10 ...
#                             evaluate_hessian=true, batch=1, devices=[0])   # ... plus batch / devices
#     initialize_states!(solver, x_guess); initialize_controls!(solver, u_guess)
#     solve!(solver); x, u = get_trajectory(solver)
#
# The constructors build the reference element (so everything of the reference keeps working on it) AND record
# the element's Symbolics expressions, emitted through Symbolics' C target (`build_function(...;
# target=Symbolics.CTarget())`), in a registry keyed by the element object. `Solver` collects them into the
# JSON model spec, has `python -m dto_b200.spec_io` compile it to a CUDA model library for sm_100a
# (content-addressed cache: the reference's "#TODO: option to load/save methods", src/dynamics.jl:22) and hands
# Ipopt a `BatchedNLPData` evaluator instead of the reference's NLPData (src/data.jl:233-234).
module DTOB200

using MathOptInterface
const MOI = MathOptInterface
using Symbolics
using SparseArrays: findnz
using LinearAlgebra: dot
import Ipopt
import DirectTrajectoryOptimization
const DTO = DirectTrajectoryOptimization

const libdto = get(ENV, "DTO_LIB", "libdto.so")
const python = get(ENV, "DTO_PYTHON", "python")
const repo   = get(ENV, "DTO_REPO", normpath(joinpath(@__DIR__, "..")))

# ---------------------------------------------------------------- thin ccall layer (include/dto.h)
check(status::Cint) = status == 0 || error("dto: " * unsafe_string(ccall((:dto_last_error, libdto), Cstring, ())))

struct ShapeDesc                       # dto_shape_desc
    T::Int32
    dynamics_kind::Ptr{Int32}
    cost_kind::Ptr{Int32}
    stage_kind::Ptr{Int32}
    use_general::Int32
    parameter_dim::Ptr{Int32}
    parameter_offset::Ptr{Int32}
    num_parameter::Int32
end

function model_load(path::String)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:dto_model_load, libdto), Cint, (Cstring, Ref{Ptr{Cvoid}}), path, h))
    h[]
end

function shape_create(model, T, kd::Vector{Int32}, kc::Vector{Int32}, ks::Vector{Int32}, use_general::Bool,
                      pdim::Vector{Int32})
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve kd kc ks pdim begin
        d = Ref(ShapeDesc(T, pointer(kd), pointer(kc), pointer(ks), use_general, pointer(pdim), C_NULL, 0))
        check(ccall((:dto_shape_create, libdto), Cint, (Ptr{Cvoid}, Ref{ShapeDesc}, Ref{Ptr{Cvoid}}), model, d, h))
    end
    h[]
end

function batch_create(shape, B::Integer, devices::Vector{Cint})
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:dto_batch_create, libdto), Cint, (Ptr{Cvoid}, Int64, Ptr{Cint}, Cint, Ref{Ptr{Cvoid}}),
                shape, B, devices, length(devices), h))
    h[]
end

num_variables(s)  = ccall((:dto_num_variables, libdto), Int64, (Ptr{Cvoid},), s)
num_constraint(s) = ccall((:dto_num_constraint, libdto), Int64, (Ptr{Cvoid},), s)
num_jacobian(s)   = ccall((:dto_num_jacobian, libdto), Int64, (Ptr{Cvoid},), s)
num_hessian(s)    = ccall((:dto_num_hessian, libdto), Int64, (Ptr{Cvoid},), s)

function structure(f::Symbol, s, n)
    r = Vector{Int64}(undef, n); c = Vector{Int64}(undef, n)
    check(ccall((f, libdto), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}), s, r, c))
    collect(zip(r, c))                  # Vector{Tuple{Int,Int}}, 1-based, reference order
end

function constraint_bounds(s)
    n = num_constraint(s)
    lo = Vector{Float64}(undef, n); up = Vector{Float64}(undef, n)
    check(ccall((:dto_constraint_bounds, libdto), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), s, lo, up))
    lo, up
end

"z-layout of the shape (src/dynamics.jl:188-195): 1-based index ranges of x_t and u_t"
function knot_layout(s, T)
    xs = Vector{Int64}(undef, T); nx = Vector{Int32}(undef, T); us = Vector{Int64}(undef, T); nu = Vector{Int32}(undef, T)
    check(ccall((:dto_knot_layout, libdto), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int32}, Ptr{Int64}, Ptr{Int32}), s, xs, nx, us, nu))
    [collect(xs[t]:xs[t] + nx[t] - 1) for t in 1:T], [collect(us[t]:us[t] + nu[t] - 1) for t in 1:T]
end

# ---------------------------------------------------------------- evaluator
mutable struct BatchedNLPData <: MOI.AbstractNLPEvaluator
    model::Ptr{Cvoid}
    shape::Ptr{Cvoid}
    batch::Ptr{Cvoid}
    B::Int
    hessian_lagrangian::Bool
    jacobian_sparsity::Vector{Tuple{Int,Int}}
    hessian_lagrangian_sparsity::Vector{Tuple{Int,Int}}
    sigma::Vector{Float64}
end

function BatchedNLPData(model_path, T, kd, kc, ks; use_general=false, pdim=zeros(Int32, T), batch=1,
                        devices=Cint[0], evaluate_hessian=false)
    m = model_load(model_path)
    s = shape_create(m, T, Int32.(kd), Int32.(kc), Int32.(ks), use_general, Int32.(pdim))
    b = batch_create(s, batch, Cint.(devices))
    BatchedNLPData(m, s, b, batch, evaluate_hessian,
                   structure(:dto_jacobian_structure, s, num_jacobian(s)),
                   structure(:dto_hessian_lagrangian_structure, s, num_hessian(s)), ones(batch))
end

set_x!(nlp, z) = check(ccall((:dto_set_x, libdto), Cint, (Ptr{Cvoid}, Ptr{Float64}), nlp.batch, z))
set_parameters!(nlp, w) = check(ccall((:dto_set_parameters, libdto), Cint, (Ptr{Cvoid}, Ptr{Float64}), nlp.batch, w))

# the five callbacks, method for method as /root/reference/src/moi.jl:1-120 (batch = 1: z is a Vector;
# batch = B: z, outputs are B x n row-major, i.e. Julia matrices of size (n, B))
function MOI.eval_objective(nlp::BatchedNLPData, z)
    set_x!(nlp, z)
    f = Vector{Float64}(undef, nlp.B)
    check(ccall((:dto_eval_objective, libdto), Cint, (Ptr{Cvoid}, Ptr{Float64}), nlp.batch, f))
    nlp.B == 1 ? f[1] : f
end
function MOI.eval_objective_gradient(nlp::BatchedNLPData, g, z)
    set_x!(nlp, z)
    check(ccall((:dto_eval_objective_gradient, libdto), Cint, (Ptr{Cvoid}, Ptr{Float64}), nlp.batch, g)); return
end
function MOI.eval_constraint(nlp::BatchedNLPData, c, z)
    set_x!(nlp, z)
    check(ccall((:dto_eval_constraint, libdto), Cint, (Ptr{Cvoid}, Ptr{Float64}), nlp.batch, c)); return
end
function MOI.eval_constraint_jacobian(nlp::BatchedNLPData, J, z)
    set_x!(nlp, z)
    check(ccall((:dto_eval_constraint_jacobian, libdto), Cint, (Ptr{Cvoid}, Ptr{Float64}), nlp.batch, J)); return
end
function MOI.eval_hessian_lagrangian(nlp::BatchedNLPData, H, z, σ, λ)
    set_x!(nlp, z)
    fill!(nlp.sigma, σ)
    check(ccall((:dto_set_duals, libdto), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), nlp.batch, nlp.sigma, λ))
    check(ccall((:dto_eval_hessian_lagrangian, libdto), Cint, (Ptr{Cvoid}, Ptr{Float64}), nlp.batch, H)); return
end
MOI.features_available(nlp::BatchedNLPData) = nlp.hessian_lagrangian ? [:Grad, :Jac, :Hess] : [:Grad, :Jac]
MOI.initialize(nlp::BatchedNLPData, features) = nothing
MOI.jacobian_structure(nlp::BatchedNLPData) = nlp.jacobian_sparsity
MOI.hessian_lagrangian_structure(nlp::BatchedNLPData) = nlp.hessian_lagrangian_sparsity

# ---------------------------------------------------------------- expression export (Symbolics C target)
"`@variables name[1:n]` as the reference's constructors write it (src/dynamics.jl:23): a Vector{Num}"
symbolic_vector(name::Symbol, n::Int) = n == 0 ? Num[] : collect(first(Symbolics.@variables $name[1:n]))

"One C function `void fname(double* out, const double* a1, ...)` for the expressions `ex` over the argument
vectors `args` named `names` -- Symbolics' own C target, zero-based references, `pow` for `^` (SURVEY App. C).
Arguments of length zero are dropped from the signature (C has no empty arrays); the parser is told the same."
function ctarget(fname::String, ex, names::Vector{Symbol}, args)
    keep = [i for i in eachindex(args) if length(args[i]) > 0]
    Symbolics.build_function(collect(ex), args[keep]...; target=Symbolics.CTarget(), fname=Symbol(fname),
                             lhsname=:out, rhsnames=names[keep], expression=Val{true})
end

sparsity_lists(S) = (I = findnz(S)[1]; J = findnz(S)[2]; [collect(Int, I), collect(Int, J)])   # CSC order, 1-based

"Re-trace `f` like Dynamics(f, ny, nx, nu; ...) does (src/dynamics.jl:23-35) and describe it for the code generator."
function dynamics_spec(f, ny, nx, nu; num_parameter=0, evaluate_hessian=false)
    y, x, u, w = symbolic_vector(:y, ny), symbolic_vector(:x, nx), symbolic_vector(:u, nu), symbolic_vector(:w, num_parameter)
    ev = f(y, x, u, w)
    d = Dict{String,Any}("num_next_state" => ny, "num_state" => nx, "num_action" => nu, "num_parameter" => num_parameter,
             "evaluate_c" => ctarget("dyn_evaluate", ev, [:y, :x, :u, :w], [y, x, u, w]),
             "jacobian_sparsity" => sparsity_lists(Symbolics.jacobian_sparsity(ev, [x; u; y])),
             "evaluate_hessian" => evaluate_hessian, "hessian_sparsity" => [Int[], Int[]])
    if evaluate_hessian
        λ = symbolic_vector(:lam, ny)
        d["hessian_sparsity"] = sparsity_lists(Symbolics.hessian_sparsity(dot(λ, ev), [x; u; y]))
    end
    d
end

"src/costs.jl:18-27: scalar cost over [x; u]; the gradient is dense (no pattern to hand over)."
function cost_spec(f, nx, nu; num_parameter=0, evaluate_hessian=false)
    x, u, w = symbolic_vector(:x, nx), symbolic_vector(:u, nu), symbolic_vector(:w, num_parameter)
    ev = [f(x, u, w)]
    d = Dict{String,Any}("num_state" => nx, "num_action" => nu, "num_parameter" => num_parameter,
             "evaluate_c" => ctarget("cost_evaluate", ev, [:x, :u, :w], [x, u, w]),
             "evaluate_hessian" => evaluate_hessian, "hessian_sparsity" => [Int[], Int[]])
    evaluate_hessian && (d["hessian_sparsity"] = sparsity_lists(Symbolics.hessian_sparsity(ev[1], [x; u])))
    d
end

"src/constraints.jl:27-40: stage constraint c(x, u, w) over [x; u]; inequality rows are local row numbers."
function constraint_spec(f, nx, nu; num_parameter=0, indices_inequality=Int[], evaluate_hessian=false)
    x, u, w = symbolic_vector(:x, nx), symbolic_vector(:u, nu), symbolic_vector(:w, num_parameter)
    ev = f(x, u, w)
    d = Dict{String,Any}("num_state" => nx, "num_action" => nu, "num_parameter" => num_parameter,
             "evaluate_c" => ctarget("stage_evaluate", ev, [:x, :u, :w], [x, u, w]),
             "jacobian_sparsity" => sparsity_lists(Symbolics.jacobian_sparsity(ev, [x; u])),
             "indices_inequality" => collect(Int, indices_inequality),
             "evaluate_hessian" => evaluate_hessian, "hessian_sparsity" => [Int[], Int[]])
    if evaluate_hessian
        λ = symbolic_vector(:lam, length(ev))
        d["hessian_sparsity"] = sparsity_lists(Symbolics.hessian_sparsity(dot(λ, ev), [x; u]))
    end
    d
end

"src/general_constraint.jl:23-36: g(z, w) over the whole trajectory z and the flat parameter vector."
function general_spec(f, nz, nw; indices_inequality=Int[], evaluate_hessian=false)
    z, w = symbolic_vector(:z, nz), symbolic_vector(:w, nw)
    ev = f(z, w)
    d = Dict{String,Any}("num_variables" => nz, "num_parameter" => nw,
             "evaluate_c" => ctarget("general_evaluate", ev, [:z, :w], [z, w]),
             "jacobian_sparsity" => sparsity_lists(Symbolics.jacobian_sparsity(ev, z)),
             "indices_inequality" => collect(Int, indices_inequality),
             "evaluate_hessian" => evaluate_hessian, "hessian_sparsity" => [Int[], Int[]])
    if evaluate_hessian
        λ = symbolic_vector(:lam, length(ev))
        d["hessian_sparsity"] = sparsity_lists(Symbolics.hessian_sparsity(dot(λ, ev), z))
    end
    d
end

# ---------------------------------------------------------------- drop-in constructors: reference element + its spec
const SPECS = IdDict{Any,Dict{String,Any}}()     # reference element object  =>  its spec for the code generator

function Dynamics(f::Function, ny::Int, nx::Int, nu::Int; num_parameter::Int=0, evaluate_hessian=false)
    el = DTO.Dynamics(f, ny, nx, nu; num_parameter=num_parameter, evaluate_hessian=evaluate_hessian)
    SPECS[el] = dynamics_spec(f, ny, nx, nu; num_parameter=num_parameter, evaluate_hessian=evaluate_hessian)
    el
end
function Cost(f::Function, nx::Int, nu::Int; num_parameter::Int=0, evaluate_hessian=false)
    el = DTO.Cost(f, nx, nu; num_parameter=num_parameter, evaluate_hessian=evaluate_hessian)
    SPECS[el] = cost_spec(f, nx, nu; num_parameter=num_parameter, evaluate_hessian=evaluate_hessian)
    el
end
function Constraint(f::Function, nx::Int, nu::Int; num_parameter::Int=0, indices_inequality=collect(1:0), evaluate_hessian=false)
    el = DTO.Constraint(f, nx, nu; num_parameter=num_parameter, indices_inequality=indices_inequality, evaluate_hessian=evaluate_hessian)
    SPECS[el] = constraint_spec(f, nx, nu; num_parameter=num_parameter, indices_inequality=indices_inequality,
                                evaluate_hessian=evaluate_hessian)
    el
end
Constraint() = DTO.Constraint()                   # empty (src/constraints.jl:66-78): kind -1, nothing to generate
function GeneralConstraint(f::Function, nz::Int, nw::Int; indices_inequality=collect(1:0), evaluate_hessian=false)
    el = DTO.GeneralConstraint(f, nz, nw; indices_inequality=indices_inequality, evaluate_hessian=evaluate_hessian)
    SPECS[el] = general_spec(f, nz, nw; indices_inequality=indices_inequality, evaluate_hessian=evaluate_hessian)
    el
end
GeneralConstraint() = DTO.GeneralConstraint()
const Bound = DTO.Bound

spec_of(el) = haskey(SPECS, el) ? SPECS[el] :
    error("DTOB200: this element was built with the reference's constructor; the CUDA backend needs its expressions -- " *
          "build it with DTOB200.Dynamics / Cost / Constraint / GeneralConstraint (arbitrary closures cannot run on the GPU, " *
          "there is no CPU fallback)")

"Distinct element objects of one role -> (kind per knot (0-based, -1 = empty), list of their specs)"
function kinds(els; empty = el -> false)
    seen = IdDict{Any,Int}(); specs = Dict{String,Any}[]; kind = Int32[]
    for el in els
        if empty(el)
            push!(kind, -1); continue
        end
        haskey(seen, el) || (push!(specs, spec_of(el)); seen[el] = length(specs) - 1)
        push!(kind, seen[el])
    end
    kind, specs
end

"The JSON model spec of a problem (spec_io.py's format) from the arguments of Solver(...) (src/solver.jl:6-10)."
function export_spec(dynamics, objective, constraints; general_constraint=DTO.GeneralConstraint(), name="model")
    T = length(objective)
    kd, sd = kinds(dynamics)
    kc, sc = kinds(objective)
    ks, ss = kinds(constraints; empty = c -> c.num_constraint == 0)
    gen = general_constraint.num_constraint == 0 ? nothing : spec_of(general_constraint)
    Dict{String,Any}("name" => name, "dynamics" => sd, "costs" => sc, "constraints" => ss, "general" => gen,
         "shape" => Dict("T" => T, "dynamics_kind" => kd, "cost_kind" => kc, "stage_kind" => ks))
end

# minimal JSON writer (no JSON.jl dependency in the reference's Project.toml)
json(x::AbstractString) = "\"" * replace(replace(replace(x, "\\" => "\\\\"), "\"" => "\\\""), "\n" => "\\n") * "\""
json(x::Bool) = x ? "true" : "false"
json(x::Nothing) = "null"
json(x::Real) = string(x)
json(x::AbstractVector) = "[" * join(json.(x), ",") * "]"
json(x::AbstractDict) = "{" * join([json(string(k)) * ":" * json(v) for (k, v) in x], ",") * "}"

"Compile (or find in the content-addressed cache) the CUDA model library of a spec; returns the path of the .so"
function build_model(spec::AbstractDict)
    path = tempname() * ".json"
    write(path, json(spec))
    strip(read(setenv(`$python -m dto_b200.spec_io $path`; dir=repo), String))
end

# ---------------------------------------------------------------- Solver: same arguments as src/solver.jl:6-10 + batch, devices
struct Solver
    nlp::BatchedNLPData
    optimizer::Ipopt.Optimizer                 # batch == 1: the one Ipopt instance (src/data.jl:237)
    variables::Vector{MOI.VariableIndex}
    state_indices::Vector{Vector{Int}}
    action_indices::Vector{Vector{Int}}
    z::Vector{Float64}                          # host mirror for get_trajectory (src/solver.jl:41-43)
    lower::Vector{Float64}                      # primal_bounds (src/data.jl:123-133): handed to dto_sqp_solve for batch > 1
    upper::Vector{Float64}
    z0::Matrix{Float64}                         # [n, batch] initial guesses of the batched solve (column b = problem b)
end

function Solver(dynamics, objective, constraints, bounds;
    evaluate_hessian=false,
    general_constraint=DTO.GeneralConstraint(),
    options=DTO.Options(),
    parameters=[[zeros(d.num_parameter) for d in dynamics]..., zeros(0)],
    batch::Int=1, devices=Cint[0], name="model")

    T = length(objective)
    spec = export_spec(dynamics, objective, constraints; general_constraint=general_constraint, name=name)
    so = build_model(spec)
    sh = spec["shape"]
    pdim = Int32[t <= length(dynamics) ? dynamics[t].num_parameter : 0 for t in 1:T]
    nlp = BatchedNLPData(String(so), T, sh["dynamics_kind"], sh["cost_kind"], sh["stage_kind"];
                         use_general=general_constraint.num_constraint > 0, pdim=pdim, batch=batch,
                         devices=Cint.(devices), evaluate_hessian=evaluate_hessian)
    w = vcat(parameters...)                                    # src/data.jl:218 layout, one copy per problem
    length(w) > 0 && set_parameters!(nlp, repeat(w, batch))
    xi, ui = knot_layout(nlp.shape, T)

    # variable bounds exactly as primal_bounds (src/data.jl:123-133)
    n = num_variables(nlp.shape)
    lower, upper = fill(-Inf, n), fill(Inf, n)
    for (t, bnd) in enumerate(bounds)
        length(bnd.state_lower)  > 0 && (lower[xi[t]] = bnd.state_lower)
        length(bnd.state_upper)  > 0 && (upper[xi[t]] = bnd.state_upper)
        length(bnd.action_lower) > 0 && (lower[ui[t]] = bnd.action_lower)
        length(bnd.action_upper) > 0 && (upper[ui[t]] = bnd.action_upper)
    end

    # SolverData (src/data.jl:222-255) with the batched evaluator in the NLP block
    clo, cup = constraint_bounds(nlp.shape)
    block = MOI.NLPBlockData(MOI.NLPBoundsPair.(clo, cup), nlp, true)
    optimizer = Ipopt.Optimizer()
    for fld in fieldnames(typeof(options))
        optimizer.options[String(fld)] = getfield(options, fld)
    end
    z = MOI.add_variables(optimizer, n)
    for i = 1:n
        MOI.add_constraint(optimizer, z[i], MOI.LessThan(upper[i]))
        MOI.add_constraint(optimizer, z[i], MOI.GreaterThan(lower[i]))
    end
    MOI.set(optimizer, MOI.NLPBlock(), block)
    MOI.set(optimizer, MOI.ObjectiveSense(), MOI.MIN_SENSE)
    Solver(nlp, optimizer, z, xi, ui, zeros(n), lower, upper, zeros(n, batch))
end

# src/solver.jl:23-47, unchanged semantics. batch == 1: the one Ipopt instance drives the callbacks (one problem per call).
# batch > 1: every problem starts from the same guess unless `problem = b` is given, and solve! runs the whole batch in
# lock step inside libdto.so (dto_sqp_solve below) -- no Ipopt, no per-problem host solver.
function DTO.initialize_states!(solver::Solver, states; problem::Int=0)
    for (t, xt) in enumerate(states), i in eachindex(xt)
        MOI.set(solver.optimizer, MOI.VariablePrimalStart(), solver.variables[solver.state_indices[t][i]], xt[i])
    end
    cols = problem == 0 ? (1:size(solver.z0, 2)) : (problem:problem)
    for (t, xt) in enumerate(states), b in cols
        solver.z0[solver.state_indices[t], b] = xt
    end
end
function DTO.initialize_controls!(solver::Solver, actions; problem::Int=0)
    for (t, ut) in enumerate(actions), j in eachindex(ut)
        MOI.set(solver.optimizer, MOI.VariablePrimalStart(), solver.variables[solver.action_indices[t][j]], ut[j])
    end
    cols = problem == 0 ? (1:size(solver.z0, 2)) : (problem:problem)
    for (t, ut) in enumerate(actions), b in cols
        solver.z0[solver.action_indices[t], b] = ut
    end
end

# ---------------------------------------------------------------- batched solve (dto_sqp_solve, include/dto.h)
"dto_sqp_options: same fields, same order (4 Int32, then 31 Float64, then 1 Int32)"
Base.@kwdef struct SQPOptions
    max_iter::Int32 = 200;  max_refactor::Int32 = 14;  max_backtrack::Int32 = 10;  soc::Int32 = 1
    tol_constraint::Float64 = 1.0e-8;  tol_dual::Float64 = 1.0e-6;  dual_reg::Float64 = 1.0e-9
    reg_first::Float64 = 1.0e-4;  reg_min::Float64 = 1.0e-20;  reg_max::Float64 = 1.0e10
    reg_inc_first::Float64 = 100.0;  reg_inc::Float64 = 8.0;  reg_dec::Float64 = 1.0 / 3.0
    armijo::Float64 = 1.0e-4;  merit_margin::Float64 = 1.1;  merit_rho::Float64 = 0.3;  merit_min::Float64 = 1.0
    lm_first::Float64 = 1.0e-2;  lm_min::Float64 = 1.0e-4;  lm_grow::Float64 = 4.0;  lm_shrink::Float64 = 0.25
    lm_grow_below::Float64 = 0.3;  lm_zero::Float64 = 1.0e-10
    lam_max::Float64 = 1.0e4;  exact_below::Float64 = 1.0
    mu_init::Float64 = 0.1;  barrier_kappa_eps::Float64 = 10.0;  barrier_kappa_mu::Float64 = 0.2;  barrier_theta_mu::Float64 = 1.5
    tau_min::Float64 = 0.99;  bound_push::Float64 = 1.0e-2;  bound_frac::Float64 = 1.0e-2;  kappa_sigma::Float64 = 1.0e10
    tiny_step::Float64 = 1.0e-6;  bound_relax::Float64 = 10.0
    hessian_approximation::Int32 = 0      # 0 exact Hessian, 1 knot-block damped BFGS (problems built with evaluate_hessian = false)
end

"""
    solve_batch(nlp, z0; lower, upper, options = SQPOptions(), lambda0 = nothing)

All problems of a one-device batch from the guesses `z0[n, B]` (column b = problem b), in lock step on the GPU: the role
Ipopt plays for one problem in `solve!(solver)` (src/solver.jl:45-47). Equality rows and rows c(z) <= 0; variables free, pinned
by `lower[i] == upper[i]`, or bounded (interior point). Returns a named tuple
`(z, lambda, iterations, converged, constraint_violation, dual_residual, objective, stats)`.
"""
function solve_batch(nlp::BatchedNLPData, z0::Matrix{Float64}; lower=nothing, upper=nothing, options::SQPOptions=SQPOptions(), lambda0=nothing)
    n, m = num_variables(nlp.shape), num_constraint(nlp.shape)
    B = size(z0, 2)
    size(z0, 1) == n || throw(DimensionMismatch("z0 must be [num_variables, batch]"))
    z, lam = Matrix{Float64}(undef, n, B), Matrix{Float64}(undef, m, B)
    its, conv = Vector{Int32}(undef, B), Vector{UInt8}(undef, B)
    cv, dr, f = Vector{Float64}(undef, B), Vector{Float64}(undef, B), Vector{Float64}(undef, B)
    stats = zeros(Int64, 16)
    lo = lower === nothing ? Ptr{Float64}(C_NULL) : pointer(lower)
    up = upper === nothing ? Ptr{Float64}(C_NULL) : pointer(upper)
    l0 = lambda0 === nothing ? Ptr{Float64}(C_NULL) : pointer(lambda0)
    GC.@preserve lower upper lambda0 begin
        check(ccall((:dto_sqp_solve, libdto), Cint,
                    (Ptr{Cvoid}, Ref{SQPOptions}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                     Ptr{Int32}, Ptr{UInt8}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}),
                    nlp.batch, Ref(options), z0, l0, lo, up, z, lam, its, conv, cv, dr, f, stats))
    end
    (z=z, lambda=lam, iterations=Int.(its), converged=conv .!= 0, constraint_violation=cv, dual_residual=dr, objective=f, stats=stats)
end

# hessian_approximation = :knot_bfgs solves a batch built without Hessians (the reference's default evaluate_hessian = false,
# which puts Ipopt in its limited-memory quasi-Newton mode) with the native solver's knot-block damped BFGS
function DTO.solve!(solver::Solver; hessian_approximation::Symbol=:exact)
    size(solver.z0, 2) == 1 && return MOI.optimize!(solver.optimizer)
    hessian_approximation in (:exact, :knot_bfgs) || throw(ArgumentError("hessian_approximation must be :exact or :knot_bfgs"))
    max_iter = Int32(get(solver.optimizer.options, "max_iter", 200))               # Options.max_iter (src/options.jl:9)
    options = SQPOptions(max_iter=max_iter, hessian_approximation=Int32(hessian_approximation === :knot_bfgs))
    solve_batch(solver.nlp, solver.z0; lower=solver.lower, upper=solver.upper, options=options)
end
"the last z any callback was handed (the reference returns its internal per-knot buffers, src/solver.jl:41-43)"
function DTO.get_trajectory(solver::Solver; problem::Int=1)
    check(ccall((:dto_get_last_x, libdto), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}), solver.nlp.batch, problem - 1, solver.z))
    T = length(solver.state_indices)
    [solver.z[solver.state_indices[t]] for t in 1:T], [solver.z[solver.action_indices[t]] for t in 1:T-1]
end

# ---------------------------------------------------------------- device-resident KKT consumer (dto_kkt_*)
# What examples/pendulum/pendulum.jl:138-211 does with the callback outputs (assemble
# [[H + primal_reg I, C'], [C, -dual_reg I]] and h = [grad + C'y; c], qdldl, solve!), for the whole
# batch on the GPU; only the solution comes back.
mutable struct BatchedKKT
    handle::Ptr{Cvoid}
    nlp::BatchedNLPData
    dim::Int
end
function BatchedKKT(nlp::BatchedNLPData; primal_reg=1.0e-5, dual_reg=1.0e-5)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:dto_kkt_create, libdto), Cint, (Ptr{Cvoid}, Cdouble, Cdouble, Ref{Ptr{Cvoid}}), nlp.batch, primal_reg, dual_reg, h))
    BatchedKKT(h[], nlp, Int(ccall((:dto_kkt_dim, libdto), Int64, (Ptr{Cvoid},), h[])))
end
"sol[dim, B] = K \\ h at (z, y) for every problem (column b = problem b; Julia is column-major, the ABI problem-major)"
function solve!(sol::Matrix{Float64}, kkt::BatchedKKT, z::Matrix{Float64}, y::Matrix{Float64})
    nlp = kkt.nlp
    check(ccall((:dto_set_x, libdto), Cint, (Ptr{Cvoid}, Ptr{Float64}), nlp.batch, z))
    fill!(nlp.sigma, 1.0)                                               # pendulum.jl:136 evaluates with sigma = 1.0
    check(ccall((:dto_set_duals, libdto), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), nlp.batch, nlp.sigma, y))
    check(ccall((:dto_kkt_solve, libdto), Cint, (Ptr{Cvoid}, Ptr{Float64}), kkt.handle, sol))
    sol
end

end # module
