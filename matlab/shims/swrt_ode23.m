function stats = swrt_ode23(eng, tspan, tmax, rtol, atol)
% stats = swrt_ode23(eng, tspan, tmax [, rtol, atol])
% Drop-in for   [~, Y] = ode23(ray_ode, [0, dt], y0)   of qgsw_raytrace.m:143-150 and
% qg2layersw_raytrace.m:189-196 with the packets RESIDENT in the engine `eng`: the three Bogacki-Shampine
% stages, ynew and the error ratio run on the device (swrt_bs23_*); only the scalar error norm comes back,
% and this controller -- the published ode23 algorithm (Shampine & Reichelt 1997) with MATLAB's defaults
% RelTol 1e-3, AbsTol 1e-6, MaxStep 0.1*|tf-t0| -- stays on the host.  alpha = t/tmax as qgsw_raytrace.m:261.
% Same logic as swraytracing_b200/reference_api.py: ode23 (which is what the test-suite exercises).
if nargin < 4, rtol = 1e-3; end
if nargin < 5, atol = 1e-6; end
t0 = tspan(1); tfinal = tspan(end);
% MATLAB's tdir: a decreasing tspan ([T 0]) integrates backward; every step is h = tdir*absh
if tfinal >= t0, tdir = 1; else, tdir = -1; end
if any(tdir * diff(tspan) < 0)
    error('swrt:ode23', 'tspan must be monotonic (an entry goes against the direction from tspan(1) to tspan(end))');
end
pw = 1/3; threshold = atol / rtol;
hmax = min(abs(tfinal - t0), abs(0.1 * (tfinal - t0)));
t = t0;
rh = swrt_mex('bs23_begin', eng, t / tmax, threshold) / (0.8 * rtol^pw);
absh = min(hmax, abs(tspan(2) - tspan(1)));          % MATLAB's htspan: the FIRST output interval bounds the initial step
if absh * rh > 1, absh = 1 / rh; end
absh = max(absh, 16 * eps(t));
nsteps = 0; nfailed = 0; done = false;
while ~done
    hmin = 16 * eps(t);
    absh = min(hmax, max(hmin, absh));
    h = tdir * absh;
    if 1.1 * absh >= abs(tfinal - t)
        h = tfinal - t; absh = abs(h); done = true;
    end
    nofailed = true;
    while true
        if done, tnew = tfinal; else, tnew = t + h; end
        err = absh * swrt_mex('bs23_attempt', eng, h, [t + 0.5 * h, t + 0.75 * h, tnew] / tmax, threshold);
        if ~(err <= rtol)
            nfailed = nfailed + 1;
            if absh <= hmin, error('swrt:ode23', 'step size below hmin at t = %g', t); end
            if nofailed
                nofailed = false;
                absh = max(hmin, absh * max(0.5, 0.8 * (rtol / err)^pw));
            else
                absh = max(hmin, 0.5 * absh);
            end
            h = tdir * absh; done = false;
        else
            break
        end
    end
    nsteps = nsteps + 1;
    swrt_mex('bs23_accept', eng);
    if nofailed
        temp = 1.25 * (err / rtol)^pw;
        if temp > 0.2, absh = absh / temp; else, absh = 5.0 * absh; end
    end
    t = tnew;
end
stats = struct('nsteps', nsteps, 'nfailed', nfailed, 't', t);
end
