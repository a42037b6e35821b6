function em_sample_b200(parameters_filename, varargin)
% EM_SAMPLE_B200  Drop-in body for em_sample.m (em_sample.m:1-104, called by RUN_1_emsample.m:38-47) that samples on a B200
% and formats the rows there too: only the text crosses PCIe, and MATLAB writes it with fwrite.  Same name-value arguments
% as em_sample.m:17-39; the same two files: initial.txt ("id <labels>" header, one row "id v1 ... vn" per sample) and
% transition.txt ("initial_id t <labels of the (t+1) variables>" header, one row "id t x_dyn..." per sample and second),
% numbers exactly as fprintf('%g') prints them (emb_mex 'em_sample_text' -> emb_format_em_sample).
% As in the Python mirror (em_model_manned_bayes_b200/em_sample.py): the prior is the intended zero prior (em_sample.m:50 sets
% 'constant', which the reference rejects at HEAD), and the random stream is the keyed stream with key rng_seed, not
% MATLAB's twister.  SOURCE ONLY (no MATLAB in the build image).
p = inputParser;
addRequired(p, 'parameters_filename', @ischar);
addParameter(p, 'initial_output_filename', 'initial.txt', @ischar);
addParameter(p, 'transition_output_filename', 'transition.txt', @ischar);
addParameter(p, 'num_initial_samples', 100, @isnumeric);
addParameter(p, 'num_transition_samples', 60, @isnumeric);
addParameter(p, 'start', {}, @iscell);
addParameter(p, 'isOverwriteZeroBoundaries', false, @islogical);
addParameter(p, 'idxZeroBoundaries', [1 2 3], @isnumeric);
addParameter(p, 'rng_seed', 42, @isnumeric);
addParameter(p, 'chunk', 65536, @isnumeric);   % tracks per GPU call: bounds the host memory of one call's text
parse(p, parameters_filename, varargin{:});
r = p.Results;

p0 = em_read(parameters_filename);             % labels and temporal_map for the header lines
h = emb_mex('load', parameters_filename, r.isOverwriteZeroBoundaries, r.idxZeroBoundaries);
cleanup = onCleanup(@() emb_mex('free', h));
opts = struct();
if ~isempty(r.start)                                                              % em_sample.m:53-55
    st = nan(1, numel(r.start));
    for i = 1:numel(r.start)
        if ~isempty(r.start{i}), st(i) = r.start{i}; end
    end
    opts.start = st;
end

fi = fopen(r.initial_output_filename, 'w');
ft = fopen(r.transition_output_filename, 'w');
fprintf(fi, 'id ');                                                               % :59-66
fprintf(fi, '%s ', p0.labels_initial{:});
fprintf(fi, '\n');
fprintf(ft, 'initial_id t ');                                                     % :68-74
fprintf(ft, '%s ', p0.labels_transition{p0.temporal_map(:, 2)});
fprintf(ft, '\n');
n = r.num_initial_samples;
T = r.num_transition_samples;
for first = 0:r.chunk:n - 1                                                       % :78-100
    [txt_i, txt_t] = emb_mex('em_sample_text', h, r.rng_seed, first, min(r.chunk, n - first), T, opts);
    fwrite(fi, txt_i, 'uint8');
    fwrite(ft, txt_t, 'uint8');
end
fclose(fi);
fclose(ft);
end
