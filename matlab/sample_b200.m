function [out_inits, out_events, out_samples, out_EME] = sample_b200(self, n_samples, sample_time, varargin)
% SAMPLE_B200  Drop-in body for UncorEncounterModel.sample (UncorEncounterModel.m:192-313) that runs the sampling on a
% B200 through emb_mex.  Same arguments ('seed', 'isQuantize500', 'layers'), same four outputs (out_EME is an array of
% EncounterModelEvents, :222,300).  Reads only properties the class has (EncounterModel.m:5-70).
% SOURCE ONLY (no MATLAB in the build image).  A maintainer replaces the body of the method by a call to this function.
p = inputParser;
addRequired(p, 'nSamples', @isnumeric);
addRequired(p, 'sample_time', @isnumeric);
addParameter(p, 'seed', nan, @isnumeric);
addParameter(p, 'isQuantize500', false, @islogical);
addParameter(p, 'layers', [], @isnumeric);
addParameter(p, 'verify', false, @islogical);   % recompute out_samples / out_EME with the reference's functions and compare
parse(p, n_samples, sample_time, varargin{:});
seed = p.Results.seed;

% rng handling of :213-216 / :310-312.  The GPU stream is keyed by (seed, sample, ...), so a given 'seed' is used as the key
% and the caller's global stream is left exactly as the reference leaves it (saved, reseeded, restored); without a seed
% one key is drawn from the caller's stream, which therefore advances as it does in the reference.
if ~isnan(seed) && ~isempty(seed)
    oldSeed = rng;
    rng(seed, 'twister');
    key = seed;
else
    key = randi(2^31 - 1);
end

idxL = find(strcmp(self.labels_initial, '"L"'));
idxV = find(strcmp(self.labels_initial, '"v"'));
idxDV = find(strcmp(self.labels_initial, '"\dot v"'));
idxDH = find(strcmp(self.labels_initial, '"\dot h"'));
idxDPsi = find(strcmp(self.labels_initial, '"\dot \psi"'));
if isempty(idxDV) || isempty(idxDH) || isempty(idxDPsi)                                    % :231-234
    error('dynvar:empty', 'Model does not have a dynamic variable for either acceleration, vertical rate, or turn rate');
end

h = emb_handle(self);
opts = struct('reject_mode', 1, 'idx_v', idxV, 'idx_dh', idxDH, 'idx_L', idxL, ...
              'is_quantize500', p.Results.isQuantize500, 'layers', p.Results.layers);
st = nan(1, self.n_initial);                                                                % bn_sample.m:45: [] / NaN = free
for i = 1:self.n_initial
    if ~isempty(self.start{i}), st(i) = self.start{i}; end
end
opts.start = st;
[events, offsets, out_inits, ~, ~, out_samples, ctl] = emb_mex('sample_events', h, key, 0, n_samples, sample_time, opts);
% events: 4 x rows [dt; var; value; bin]; rows offsets(ii)+1 : offsets(ii+1) are out_events{ii} of
% dbn_hierarchical_sample.m:9-37, built on the GPU in the reference's own row order.  out_samples{ii} and ctl{ii} (the
% event matrix of :286-297) are computed on the GPU from the same rows with the same fp64 operations as the reference's
% per-track statements; 'verify', true recomputes them with those statements and requires them to be identical.

out_events = cell(n_samples, 1);
out_EME(n_samples, 1) = EncounterModelEvents;                                               % :222
tm = self.temporal_map;
idxEME = [find(tm(:, 1) == idxDH), find(tm(:, 1) == idxDPsi), find(tm(:, 1) == idxDV)] + 1; % :291
for ii = 1:n_samples
    out_events{ii} = events(1:3, offsets(ii) + 1:offsets(ii + 1))';
    out_EME(ii) = EncounterModelEvents('event', ctl{ii});                                  % :300
    if p.Results.verify
        controls = events2controls(out_inits(ii, :), out_events{ii}, struct('temporal_map', tm));   % :286
        controls = controls(:, [1 idxEME]);                                                 % :292
        controls(:, 2) = controls(:, 2) / 60;                                               % :295
        controls(:, 3) = deg2rad(controls(:, 3));                                           % :296
        controls(:, 4) = controls(:, 4) * 1.68780972222222;                                 % :297
        assert(isequal(out_samples{ii}, events2samples(out_inits(ii, :), out_events{ii})) && ...
               isequal(ctl{ii}, controls), 'sample_b200: GPU out_samples / out_EME differ from the reference (track %d)', ii);
    end
end

if ~isnan(seed) && ~isempty(seed)
    rng(oldSeed);                                                                           % :310-312
end
end
