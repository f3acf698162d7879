classdef TinyMPC < handle
    % TinyMPC  MATLAB front end of the B200-native batched TinyMPC solver.
    %
    % Same public surface as the reference class (reference src/TinyMPC.m:42-325: setup, set_x0,
    % set_x_ref, set_u_ref, update_settings, solve, get_solution, set_bound_constraints,
    % set_linear_constraints, set_cone_constraints, set_equality_constraints,
    % set_sensitivity_matrices, compute_cache_terms, compute_sensitivity_autograd, reset) so that
    % existing scripts run unchanged; every solve executes on the GPU through the MEX gateway
    % tinympc_matlab (matlab/bindings.cpp).  New: solve_batch, set_option, get_stats.

    properties
        nx = 0; nu = 0; N = 0;
        A = []; B = []; Q = []; R = [];
        rho = 1.0;
        is_setup = false;
        settings = struct();
        x_min = []; x_max = []; u_min = []; u_max = [];
        dK = []; dP = []; dC1 = []; dC2 = [];
        session_size = 0;      % number of warm-started GPU copies of this solver (session_create), 0 = none
    end

    methods
        function obj = TinyMPC()
            % defaults of the reference class (src/TinyMPC.m:26-39)
            names  = {'abs_pri_tol','abs_dua_tol','max_iter','check_termination','en_state_bound','en_input_bound', ...
                      'en_state_soc','en_input_soc','en_state_linear','en_input_linear','adaptive_rho', ...
                      'adaptive_rho_min','adaptive_rho_max','adaptive_rho_enable_clipping'};
            values = {1e-4, 1e-4, 100, 1, false, false, false, false, false, false, false, 0.1, 10.0, true};
            obj.settings = cell2struct(values(:), names(:), 1);
        end

        function setup(obj, A, B, Q, R, N, varargin)
            % setup(A, B, Q, R, N, 'rho', 1.0, 'fdyn', f, 'max_iter', 100, ...)
            assert(size(A,1) == size(A,2), 'A must be square');
            assert(size(A,1) == size(B,1), 'A and B row dimensions must match');
            assert(size(Q,1) == size(A,1), 'Q must match A dimensions');
            assert(size(R,1) == size(B,2), 'R must match B column dimension');
            assert(N >= 2, 'N must be >= 2');
            obj.nx = size(A,1); obj.nu = size(B,2); obj.N = N;
            obj.A = A; obj.B = B; obj.Q = Q; obj.R = R;

            opts = struct('rho', 1.0, 'fdyn', [], 'verbose', false, 'abs_pri_tol', 1e-4, 'abs_dua_tol', 1e-4, ...
                          'max_iter', 100, 'check_termination', 1, 'en_state_bound', false, 'en_input_bound', false, ...
                          'adaptive_rho', false, 'adaptive_rho_min', 0.1, 'adaptive_rho_max', 10.0, ...
                          'adaptive_rho_enable_clipping', true);
            opts = obj.merge_known(opts, varargin{:});
            obj.rho = opts.rho;
            for f = {'abs_pri_tol','abs_dua_tol','max_iter','check_termination','adaptive_rho', ...
                     'adaptive_rho_min','adaptive_rho_max','adaptive_rho_enable_clipping'}
                obj.settings.(f{1}) = opts.(f{1});
            end
            obj.settings.en_state_bound = false;    % bounds are enabled by set_bound_constraints only
            obj.settings.en_input_bound = false;
            fdyn = opts.fdyn;
            if isempty(fdyn), fdyn = zeros(obj.nx, 1); end

            status = tinympc_matlab('setup', A, B, fdyn, Q, R, obj.rho, obj.nx, obj.nu, obj.N, opts.verbose);
            if status ~= 0
                error('TinyMPC:SetupFailed', 'Setup failed with status %d', status);
            end
            obj.is_setup = true;
            obj.push_settings();
            if opts.verbose
                fprintf('TinyMPC solver setup successful (nx=%d, nu=%d, N=%d)\n', obj.nx, obj.nu, obj.N);
            end
        end

        function set_x0(obj, x0)
            obj.require_setup();
            tinympc_matlab('set_x0', x0(:), false);
        end

        function set_x_ref(obj, x_ref)
            obj.require_setup();
            tinympc_matlab('set_x_ref', obj.spread(x_ref, obj.nx, obj.N), false);
        end

        function set_u_ref(obj, u_ref)
            obj.require_setup();
            tinympc_matlab('set_u_ref', obj.spread(u_ref, obj.nu, obj.N-1), false);
        end

        function update_settings(obj, varargin)
            obj.require_setup();
            for k = 1:2:numel(varargin)
                if isfield(obj.settings, varargin{k}), obj.settings.(varargin{k}) = varargin{k+1}; end
            end
            obj.push_settings();
        end

        function status = solve(obj)
            % One solve with the warm-start semantics of the reference (the workspace persists on the host
            % side between calls).  Returns 0 like the reference class; see get_stats for iter / status.
            obj.require_setup();
            tinympc_matlab('solve', false);
            status = 0;
        end

        function solution = get_solution(obj)
            obj.require_setup();
            [xs, us] = tinympc_matlab('get_solution', false);
            solution = struct('states', xs, 'controls', us);
        end

        function stats = get_stats(obj)
            obj.require_setup();
            [it, st, px, pu] = tinympc_matlab('get_stats', false);
            stats = struct('iter', it, 'status', st, 'primal_residual_state', px, 'primal_residual_input', pu);
        end

        function out = solve_batch(obj, X0, Xref, Uref, varargin)
            % out = solve_batch(X0, Xref, Uref)                          shared family bounds
            % out = solve_batch(X0, Xref, Uref, xmin, xmax, umin, umax)  per-problem bounds
            %   X0   nx x B
            %   Xref nx x N x B, or nx x N / nx x 1 / scalar (shared, expanded like set_x_ref), or []
            %   Uref nu x (N-1) x B, same conventions
            % Solves B independent problems of this family (cold start each) in one GPU call.
            % out.states nx x N x B, out.controls nu x (N-1) x B (single), out.iter, out.status (int32),
            % out.residuals 4 x B, out.rho B x 1.  double or single inputs; single avoids a conversion copy.
            obj.require_setup();
            B = size(X0, 2);
            Xref = obj.batch_traj(Xref, obj.nx, obj.N, B);
            Uref = obj.batch_traj(Uref, obj.nu, obj.N-1, B);
            bnd = {[], [], [], []};
            if numel(varargin) == 4
                dims = {obj.nx, obj.nx, obj.nu, obj.nu}; steps = {obj.N, obj.N, obj.N-1, obj.N-1};
                for k = 1:4, bnd{k} = obj.batch_traj(varargin{k}, dims{k}, steps{k}, B); end
            elseif ~isempty(varargin)
                error('TinyMPC:InvalidInput', 'per-problem bounds need xmin, xmax, umin, umax');
            end
            [xs, us, it, st, res, rho_out] = tinympc_matlab('solve_batch', X0, Xref, Uref, bnd{:}, false);
            out = struct('states', xs, 'controls', us, 'iter', it, 'status', st, 'residuals', res, 'rho', rho_out);
        end

        function out = solve_batch_models(obj, X0, Xref, Uref, models)
            % out = solve_batch_models(X0, Xref, Uref, models)
            % B independent problems that each bring their OWN model: what a loop of setup + solve over solvers with
            % different dynamics and costs computes, in one GPU call.  This object supplies the horizon, the settings and
            % the shared bounds and constraints; X0, Xref, Uref as for solve_batch.  models is a struct of double arrays,
            % one page per problem:
            %   A nx x nx x B, B nx x nu x B, Q nx x B, R nu x B (diag + rho, as setup stores them), rho 1 x B,
            %   Kinf nu x nx x B, Pinf nx x nx x B, Quu_inv nu x nu x B, AmBKt nx x nx x B (the cache of each model),
            %   optional f, APf (nx x B), BPf (nu x B), and dKinf, dPinf (required with adaptive rho).
            % Returns the fields of solve_batch.
            obj.require_setup();
            B = size(X0, 2);
            Xref = obj.batch_traj(Xref, obj.nx, obj.N, B);
            Uref = obj.batch_traj(Uref, obj.nu, obj.N-1, B);
            if ~isstruct(models)
                error('TinyMPC:InvalidInput', 'models must be a struct of per-problem model arrays');
            end
            names = {'A', 'B', 'f', 'Q', 'R', 'rho', 'Kinf', 'Pinf', 'Quu_inv', 'AmBKt', 'APf', 'BPf', 'dKinf', 'dPinf'};
            arrs = cell(1, numel(names));
            for k = 1:numel(names)
                if isfield(models, names{k}), arrs{k} = double(models.(names{k})); else, arrs{k} = []; end
            end
            [xs, us, it, st, res, rho_out] = tinympc_matlab('solve_batch_models', X0, Xref, Uref, arrs{:}, false);
            out = struct('states', xs, 'controls', us, 'iter', it, 'status', st, 'residuals', res, 'rho', rho_out);
        end

        function set_option(obj, name, value)
            % 'precision' 32 (fast, default for batches) | 64 (iteration counts identical to the CPU reference),
            % 'mixed' (band: fp32 pass + fp64 re-solve of the borderline problems), 'chunks', 'ctas_per_sm', 'force_wpp'
            obj.require_setup();
            tinympc_matlab('set_option', name, value);
        end

        % ---- sessions: B warm-started copies of this solver on the GPU (closed loops, examples/cartpole_example_mpc.m:36-44,
        % for B systems at once).  Constraints, settings and options are taken as they are when the session is created.
        function session_create(obj, B)
            obj.require_setup();
            tinympc_matlab('session_create', B);
            obj.session_size = B;
        end

        function session_set_x0(obj, X0)
            % X0: nx x B
            obj.require_session();
            tinympc_matlab('session_set_x0', double(X0));
        end

        function session_set_x_ref(obj, Xref)
            % Xref: nx x N x B, or nx x N / nx x 1 / scalar (shared by all problems, expanded like set_x_ref)
            obj.require_session();
            tinympc_matlab('session_set_x_ref', obj.session_traj(Xref, obj.nx, obj.N));
        end

        function session_set_u_ref(obj, Uref)
            obj.require_session();
            tinympc_matlab('session_set_u_ref', obj.session_traj(Uref, obj.nu, obj.N-1));
        end

        function session_solve(obj)
            obj.require_session();
            tinympc_matlab('session_solve');
        end

        function session_step(obj, use_solution)
            % x0 <- A x0 + B u0 + f on the GPU; u0 = work.u(:,1) (default) or the clamped solution u(:,1) (use_solution = true)
            obj.require_session();
            if nargin < 2, use_solution = false; end
            tinympc_matlab('session_step', double(use_solution));
        end

        function v = session_read(obj, field)
            % 'x0' | 'x' | 'sol_x' | 'u' | 'sol_u' | 'iter' | 'status' | 'rho' | 'residuals'
            obj.require_session();
            v = tinympc_matlab('session_read', field);
        end

        function session_destroy(obj)
            tinympc_matlab('session_destroy');
            obj.session_size = 0;
        end

        function codegen(obj, output_dir)
            % Generate the standalone project data (tiny_data.cpp/.hpp, tiny_main.cpp) + the B200 family table
            obj.require_setup();
            status = tinympc_matlab('codegen', output_dir, false);
            if status ~= 0
                error('TinyMPC:CodegenFailed', 'Code generation failed with status: %d', status);
            end
            fprintf('Code generation completed successfully in: %s\n', output_dir);
        end

        function codegen_with_sensitivity(obj, output_dir, dK, dP, dC1, dC2)
            obj.require_setup();
            obj.set_sensitivity_matrices(dK, dP, dC1, dC2);
            status = tinympc_matlab('codegen_with_sensitivity', output_dir, dK, dP, dC1, dC2, false);
            if status ~= 0
                error('TinyMPC:CodegenWithSensitivityFailed', 'Code generation with sensitivity failed with status: %d', status);
            end
            fprintf('Code generation with sensitivity matrices completed successfully in: %s\n', output_dir);
        end

        function set_sensitivity_matrices(obj, dK, dP, dC1, dC2)
            obj.require_setup();
            obj.check_sensitivity_sizes(dK, dP, dC1, dC2);
            obj.dK = dK; obj.dP = dP; obj.dC1 = dC1; obj.dC2 = dC2;
            tinympc_matlab('set_sensitivity_matrices', dK, dP, dC1, dC2, false);
        end

        function [Kinf, Pinf, Quu_inv, AmBKt] = compute_cache_terms(obj)
            % MATLAB-side Riccati iteration (single +rho, Pinf seeded with Q), as the reference class does
            obj.require_setup();
            [Kinf, Pinf, Quu_inv, AmBKt] = obj.riccati(obj.rho, obj.Q);
        end

        function [dK, dP, dC1, dC2] = compute_sensitivity_autograd(obj)
            % forward differences in rho with step 1e-6
            obj.require_setup();
            h = 1e-6;
            [K0, P0, C10, C20] = obj.lqr_terms(obj.rho);
            [K1, P1, C11, C21] = obj.lqr_terms(obj.rho + h);
            dK = (K1 - K0) / h; dP = (P1 - P0) / h; dC1 = (C11 - C10) / h; dC2 = (C21 - C20) / h;
        end

        function set_linear_constraints(obj, Alin_x, blin_x, Alin_u, blin_u)
            obj.require_setup();
            tinympc_matlab('set_linear_constraints', Alin_x, blin_x, Alin_u, blin_u, false);
            obj.settings.en_state_linear = ~isempty(Alin_x) && ~isempty(blin_x);
            obj.settings.en_input_linear = ~isempty(Alin_u) && ~isempty(blin_u);
            if obj.settings.en_state_linear || obj.settings.en_input_linear, obj.push_settings(); end
        end

        function set_bound_constraints(obj, x_min, x_max, u_min, u_max)
            obj.require_setup();
            big = 1e17;
            obj.x_min = obj.spread_bound(x_min, obj.nx, obj.N, -big);
            obj.x_max = obj.spread_bound(x_max, obj.nx, obj.N, +big);
            obj.u_min = obj.spread_bound(u_min, obj.nu, obj.N-1, -big);
            obj.u_max = obj.spread_bound(u_max, obj.nu, obj.N-1, +big);
            tinympc_matlab('set_bound_constraints', obj.x_min, obj.x_max, obj.u_min, obj.u_max, false);
            obj.settings.en_state_bound = true;
            obj.settings.en_input_bound = true;
            obj.push_settings();
        end

        function set_cone_constraints(obj, Acx, qcx, cx, Acu, qcu, cu)
            % state cones first, then input cones (as in the reference class)
            obj.require_setup();
            if ~isempty(Acx), Acx = int32(Acx(:)); qcx = int32(qcx(:)); cx = double(cx(:)); end
            if ~isempty(Acu), Acu = int32(Acu(:)); qcu = int32(qcu(:)); cu = double(cu(:)); end
            tinympc_matlab('set_cone_constraints', Acx, qcx, cx, Acu, qcu, cu, false);
            obj.settings.en_state_soc = ~isempty(Acx) && ~isempty(qcx) && ~isempty(cx);
            obj.settings.en_input_soc = ~isempty(Acu) && ~isempty(qcu) && ~isempty(cu);
            if obj.settings.en_state_soc || obj.settings.en_input_soc, obj.push_settings(); end
        end

        function set_equality_constraints(obj, Aeq_x, beq_x, Aeq_u, beq_u)
            % Aeq * x == beq expressed as the inequality pair  Aeq x <= beq,  -Aeq x <= -beq
            obj.require_setup();
            [Ax, bx] = obj.two_sided(Aeq_x, beq_x);
            [Au, bu] = obj.two_sided(Aeq_u, beq_u);
            obj.set_linear_constraints(Ax, bx, Au, bu);
        end

        function reset(obj)
            if obj.is_setup
                tinympc_matlab('reset', false);
                obj.is_setup = false;
            end
        end
    end

    methods (Access = private)
        function require_setup(obj)
            if ~obj.is_setup
                error('TinyMPC:NotSetup', 'Solver not setup. Call setup() first.');
            end
        end

        function require_session(obj)
            obj.require_setup();
            if obj.session_size < 1
                error('TinyMPC:NotSetup', 'No session. Call session_create(B) first.');
            end
        end

        function T = session_traj(obj, v, dim, steps)
            % dim x steps x B stays as it is; anything 2-D is one trajectory shared by all problems
            if ndims(v) == 3
                assert(isequal(size(v), [dim, steps, obj.session_size]), 'batched trajectory must be %d x %d x %d', dim, steps, obj.session_size);
                T = double(v);
            else
                T = double(obj.spread(v, dim, steps));
            end
        end

        function push_settings(obj)
            s = obj.settings;
            tinympc_matlab('update_settings', s.abs_pri_tol, s.abs_dua_tol, s.max_iter, s.check_termination, ...
                s.en_state_bound, s.en_input_bound, s.en_state_soc, s.en_input_soc, s.en_state_linear, s.en_input_linear, ...
                s.adaptive_rho, s.adaptive_rho_min, s.adaptive_rho_max, s.adaptive_rho_enable_clipping, false);
        end

        function opts = merge_known(~, opts, varargin)
            for k = 1:2:numel(varargin)
                if k+1 <= numel(varargin) && isfield(opts, varargin{k}), opts.(varargin{k}) = varargin{k+1}; end
            end
        end

        function M = spread(~, v, dim, steps)
            % scalar / dim x 1 / 1 x dim -> dim x steps; anything else is taken as already full
            if isscalar(v)
                M = v * ones(dim, steps);
            elseif isequal(size(v), [dim, 1])
                M = repmat(v, 1, steps);
            elseif isequal(size(v), [1, dim])
                M = repmat(v', 1, steps);
            else
                M = v;
            end
        end

        function M = spread_bound(obj, v, dim, steps, default_value)
            if isempty(v)
                M = default_value * ones(dim, steps);
            else
                M = obj.spread(v, dim, steps);
            end
        end

        function T = batch_traj(obj, v, dim, steps, B)
            % [] stays [] (zeros on the GPU side); 2-D inputs are shared by every problem
            if isempty(v)
                T = [];
            elseif ndims(v) == 3
                assert(isequal(size(v), [dim, steps, B]), 'batched trajectory must be %d x %d x %d', dim, steps, B);
                T = v;
            else
                T = repmat(obj.spread(v, dim, steps), 1, 1, B);
            end
        end

        function [Aio, bio] = two_sided(~, Aeq, beq)
            Aio = []; bio = [];
            if ~isempty(Aeq)
                beq = beq(:);
                Aio = [Aeq; -Aeq];
                bio = [beq; -beq];
            end
        end

        function [K, P, C1, C2] = riccati(obj, rho_val, P0)
            Qr = obj.Q + rho_val * eye(obj.nx);
            Rr = obj.R + rho_val * eye(obj.nu);
            K = zeros(obj.nu, obj.nx); P = P0;
            for it = 1:5000
                Kprev = K;
                K = (Rr + obj.B' * P * obj.B + 1e-8 * eye(obj.nu)) \ (obj.B' * P * obj.A);
                P = Qr + obj.A' * P * (obj.A - obj.B * K);
                if it > 1 && norm(K - Kprev) < 1e-10, break; end
            end
            C1 = inv(Rr + obj.B' * P * obj.B);
            C2 = (obj.A - obj.B * K)';
        end

        function [K, P, C1, C2] = lqr_terms(obj, rho_val)
            Qr = obj.Q + rho_val * eye(obj.nx);
            Rr = obj.R + rho_val * eye(obj.nu);
            try
                [P, Kd] = idare(obj.A, obj.B, Qr, Rr);
                K = -Kd;                       % same sign convention as the reference helper (src/TinyMPC.m:347-348)
                C1 = inv(Rr + obj.B' * P * obj.B);
                C2 = (obj.A - obj.B * K)';
            catch
                [K, P, C1, C2] = obj.riccati(rho_val, Qr);
            end
        end

        function check_sensitivity_sizes(obj, dK, dP, dC1, dC2)
            assert(isequal(size(dK), [obj.nu, obj.nx]), 'dK must be nu x nx');
            assert(isequal(size(dP), [obj.nx, obj.nx]), 'dP must be nx x nx');
            assert(isequal(size(dC1), [obj.nu, obj.nu]), 'dC1 must be nu x nu');
            assert(isequal(size(dC2), [obj.nx, obj.nx]), 'dC2 must be nx x nx');
        end
    end
end
