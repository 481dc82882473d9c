# lrcn_b200.jl -- ccall shim that swaps the hot path of lrcn.jl for liblrcn_b200.so.
#
# UNEXECUTED IN THIS REPO'S CI: Julia is not installed in the build image.  The executable mirror,
# with the same argument order for every symbol, is long-term-recurrent-convolutional-nn_b200/abi.py.
# Written in the reference's Julia-0.5 dialect (lrcn.jl uses `Array(Any,n)`, `type`, `srand`).
#
# Usage inside lrcn.jl (see INTEGRATION.md for the exact diff):
#     include("lrcn_b200.jl"); using LRCNB200
#     net = LRCNB200.create(o[:embed], o[:hidden], vocab_size, o[:batchsize])
#     LRCNB200.set_model!(net, model)                     # after initweights / JLD load   (lrcn.jl:87,90)
#     LRCNB200.load_features!(net, 0, feats); LRCNB200.load_features!(net, 1, featsvl)   # (lrcn.jl:121-123)
#     loss = LRCNB200.train_step!(net, 0, input_ids[b], sequence, index:index+l-1; pdrop=pdrop)   # (lrcn.jl:378+394)
#     model = LRCNB200.get_model(net)                     # before save(...)               (lrcn.jl:185,230)
module LRCNB200

const lib = get(ENV, "LRCN_B200_LIB", "liblrcn_b200.so")

type Config          # mirrors lrcn_config in include/lrcn_b200.h, field for field
    embed::Int32; hidden1::Int32; hidden2::Int32; vocab::Int32
    max_batch::Int32; max_len::Int32; max_gen_rows::Int32; device::Int32
    precision::Int32; use_graphs::Int32
    lr::Float64; beta1::Float64; beta2::Float64; eps::Float64
    n_gpus::Int32                        # 0/1: one GPU; 2..8: the library drives device_ids[1:n_gpus] itself
    device_ids::NTuple{8,Int32}
end

type Net
    handle::Ptr{Void}
    vocab::Int
end

lasterror() = unsafe_string(ccall((:lrcn_last_error, lib), Cstring, ()))
check(rc) = rc == 0 ? nothing : error(lasterror())     # reference convention: error(msg)
abi_version() = ccall((:lrcn_abi_version, lib), Cint, ())

function default_config()
    c = Ref(Config(0,0,0,0,0,0,0,0,0,0,0.0,0.0,0.0,0.0,0,ntuple(i->Int32(0),8)))
    check(ccall((:lrcn_config_default, lib), Cint, (Ptr{Config},), c))
    return c[]
end

# gpus: vector of CUDA ordinals.  One entry = one GPU.  Several = single-process data parallelism: lrcn.jl stays ONE
# process with ONE net; train_step!/loss take the GLOBAL batch (batchsize = global rows) and the library shards the rows,
# exchanges gradients over NVLink peer memory and shards beam search by image -- no launcher, no MPI.
# gclip: Knet Adam(gclip=...) per parameter tensor (set_gclip!); 0 = off, which is what the reference trains with.
function create(embed, hidden, vocab_size, batchsize; max_len=28, max_gen_rows=1024, gpus=[0], precision=1, gclip=0.0)
    c = default_config()
    c.embed = embed; c.hidden1 = hidden[1]; c.hidden2 = hidden[2]; c.vocab = vocab_size
    c.max_batch = batchsize; c.max_len = max_len; c.max_gen_rows = max_gen_rows
    c.device = gpus[1]; c.precision = precision
    c.n_gpus = length(gpus)
    c.device_ids = ntuple(i -> Int32(i <= length(gpus) ? gpus[i] : 0), 8)
    h = Ref{Ptr{Void}}(C_NULL)
    check(ccall((:lrcn_create, lib), Cint, (Ptr{Config}, Ptr{Ptr{Void}}), Ref(c), h))
    net = Net(h[], vocab_size)
    finalizer(net, n -> ccall((:lrcn_destroy, lib), Cint, (Ptr{Void},), n.handle))
    gclip > 0 && set_gclip!(net, gclip)
    return net
end

function param_shape(net, k)
    r = Ref{Int64}(0); c = Ref{Int64}(0)
    check(ccall((:lrcn_param_shape, lib), Cint, (Ptr{Void}, Cint, Ptr{Int64}, Ptr{Int64}), net.handle, k, r, c))
    return (Int(r[]), Int(c[]))
end

# model = the 9-element Any vector of lrcn.jl:489-510, column-major Float32 (Array, not KnetArray)
function set_model!(net, model)
    for k = 1:9
        w = convert(Array{Float32}, model[k])
        check(ccall((:lrcn_set_param, lib), Cint, (Ptr{Void}, Cint, Ptr{Float32}, Int64, Int64),
                    net.handle, k, w, size(w,1), size(w,2)))
    end
end

function getmats(sym, net, pre...)
    out = Array(Any, 9)
    for k = 1:9
        r, c = param_shape(net, k)
        w = Array(Float32, r, c)
        if sym == :param
            check(ccall((:lrcn_get_param, lib), Cint, (Ptr{Void}, Cint, Ptr{Float32}, Int64, Int64), net.handle, k, w, r, c))
        elseif sym == :grad
            check(ccall((:lrcn_get_grad, lib), Cint, (Ptr{Void}, Cint, Ptr{Float32}, Int64, Int64), net.handle, k, w, r, c))
        else
            check(ccall((:lrcn_get_adam_state, lib), Cint, (Ptr{Void}, Cint, Cint, Ptr{Float32}, Int64, Int64), net.handle, k, pre[1], w, r, c))
        end
        out[k] = w
    end
    return out
end
get_model(net) = getmats(:param, net)
get_grads(net) = getmats(:grad, net)
get_adam_state(net, which) = getmats(:adam, net, which)

function set_adam_state!(net, which, mats)
    for k = 1:9
        w = convert(Array{Float32}, mats[k])
        check(ccall((:lrcn_set_adam_state, lib), Cint, (Ptr{Void}, Cint, Cint, Ptr{Float32}, Int64, Int64),
                    net.handle, k, which, w, size(w,1), size(w,2)))
    end
end
function adam_step(net)
    t = Ref{Int64}(0)
    check(ccall((:lrcn_get_adam_step, lib), Cint, (Ptr{Void}, Ptr{Int64}), net.handle, t)); return t[]
end
set_adam_step!(net, t) = check(ccall((:lrcn_set_adam_step, lib), Cint, (Ptr{Void}, Int64), net.handle, t))

# feats::Dict{Int,Array{Float32}} exactly as loaded at lrcn.jl:121-123
function load_features!(net, split, feats)
    ids = collect(Int64, keys(feats))
    mat = Array(Float32, 4096, length(ids))          # column j = image j  => 4096 contiguous floats per image
    for (j, id) in enumerate(ids); mat[:, j] = vec(feats[id]); end
    check(ccall((:lrcn_load_features, lib), Cint, (Ptr{Void}, Cint, Ptr{Int64}, Ptr{Float32}, Int64),
                net.handle, split, ids, mat, length(ids)))
end

# sequence[t][i] (Vector of Vector{Int}) and range -> the l x B time-major matrix the ABI takes:
# tokens[t*B+i] in C order == column-major B x l matrix with tok[i,t]
function tokmat(sequence, range)
    B = length(sequence[first(range)])
    tok = Array(Int64, B, length(range))
    for (k, t) in enumerate(range); tok[:, k] = sequence[t]; end
    return tok
end

function loss(net, split, ids, sequence, range)      # replaces loss(...) lrcn.jl:553-581 / :452-474
    tok = tokmat(sequence, range); s = Ref{Float64}(0); n = Ref{Int64}(0)
    check(ccall((:lrcn_loss, lib), Cint, (Ptr{Void}, Cint, Ptr{Int64}, Ptr{Int64}, Cint, Cint, Ptr{Float64}, Ptr{Int64}),
                net.handle, split, convert(Vector{Int64}, ids), tok, size(tok,2), size(tok,1), s, n))
    return (s[], n[])                                # total log-prob and count: loss = -total/count
end

function lossgradient(net, split, ids, sequence, range; pdrop=0.0, seed=0)   # lrcn.jl:378,583
    tok = tokmat(sequence, range); l = Ref{Float64}(0)
    check(ccall((:lrcn_grad, lib), Cint, (Ptr{Void}, Cint, Ptr{Int64}, Ptr{Int64}, Cint, Cint, Cfloat, UInt64, Ptr{Float64}),
                net.handle, split, convert(Vector{Int64}, ids), tok, size(tok,2), size(tok,1), pdrop, seed, l))
    return get_grads(net)
end

update!(net) = check(ccall((:lrcn_adam_update, lib), Cint, (Ptr{Void},), net.handle))   # lrcn.jl:394

# Adam(gclip=o[:gclip]) (lrcn.jl:44-45,402): each of the 9 gradients is scaled to norm g when its norm exceeds g; 0 = off.
# One GPU only.  grad_norms: the 9 norms of the gradients currently held, computed on the device.
set_gclip!(net, g) = check(ccall((:lrcn_set_gclip, lib), Cint, (Ptr{Void}, Float64), net.handle, g))
function grad_norms(net)
    n = zeros(Float64, 9)
    check(ccall((:lrcn_grad_norms, lib), Cint, (Ptr{Void}, Ptr{Float64}), net.handle, n)); return n
end

function train_step!(net, split, ids, sequence, range; pdrop=0.0, seed=0)   # lrcn.jl:378 + :394 fused
    tok = tokmat(sequence, range); l = Ref{Float64}(0)
    check(ccall((:lrcn_train_step, lib), Cint, (Ptr{Void}, Cint, Ptr{Int64}, Ptr{Int64}, Cint, Cint, Cfloat, UInt64, Ptr{Float64}),
                net.handle, split, convert(Vector{Int64}, ids), tok, size(tok,2), size(tok,1), pdrop, seed, l))
    return l[]
end

# One epoch of the hot loop of train1 (lrcn.jl:351-396) in ONE call: `sequence`, `input_ids`, `lengths` are what minibatch()
# returned (lrcn.jl:257-297), `order` the shuffled batch starts `shuffle(1:batchsize:length(lengths))` of lrcn.jl:351.  The
# library uploads the epoch once, stages every batch on the device and skips l > 28 batches like lrcn.jl:353.
function train_epoch!(net, split, sequence, input_ids, lengths, batchsize, order; pdrop=0.0, seed=0)
    seq = convert(Matrix{Int64}, hcat(sequence...))        # B x n_rows, column-major = the C side's [n_rows][B]
    ids = convert(Matrix{Int64}, hcat(input_ids...))       # B x n_batches
    blens = convert(Vector{Int64}, lengths[1:batchsize:end])
    ord = convert(Vector{Int64}, [div(t - 1, batchsize) for t in order])   # 0-based batch numbers
    losses = zeros(Float64, length(ord)); steps = Ref{Int64}(0)
    check(ccall((:lrcn_train_epoch, lib), Cint,
                (Ptr{Void}, Cint, Ptr{Int64}, Int64, Ptr{Int64}, Ptr{Int64}, Int64, Cint, Ptr{Int64}, Int64, Cfloat, UInt64, Ptr{Float64}, Ptr{Int64}),
                net.handle, split, seq, size(seq,2), ids, blens, length(blens), size(ids,1), ord, length(ord), pdrop, seed, losses, steps))
    return losses[1:steps[]]
end

# average_loss (lrcn.jl:407-486) over a whole split in one call; returns -sum(logp)/count like the reference
function average_loss(net, split, sequence, input_ids, lengths, batchsize)
    seq = convert(Matrix{Int64}, hcat(sequence...)); ids = convert(Matrix{Int64}, hcat(input_ids...))
    blens = convert(Vector{Int64}, lengths[1:batchsize:end]); s = Ref{Float64}(0); n = Ref{Int64}(0)
    check(ccall((:lrcn_loss_epoch, lib), Cint, (Ptr{Void}, Cint, Ptr{Int64}, Int64, Ptr{Int64}, Ptr{Int64}, Int64, Cint, Ptr{Float64}, Ptr{Int64}),
                net.handle, split, seq, size(seq,2), ids, blens, length(blens), size(ids,1), s, n))
    return -s[] / n[]
end

function token_logps(net, l, B)
    out = Array(Float32, B, l+1)
    check(ccall((:lrcn_get_token_logps, lib), Cint, (Ptr{Void}, Ptr{Float32}, Int64), net.handle, out, length(out)))
    return out
end

function stage_batch!(net, slot, split, ids, sequence, range)
    tok = tokmat(sequence, range)
    check(ccall((:lrcn_stage_batch, lib), Cint, (Ptr{Void}, Cint, Cint, Ptr{Int64}, Ptr{Int64}, Cint, Cint),
                net.handle, slot, split, convert(Vector{Int64}, ids), tok, size(tok,2), size(tok,1)))
end
function train_step_staged!(net, slot; pdrop=0.0, seed=0)
    l = Ref{Float64}(0)
    check(ccall((:lrcn_train_step_staged, lib), Cint, (Ptr{Void}, Cint, Cfloat, UInt64, Ptr{Float64}), net.handle, slot, pdrop, seed, l))
    return l[]
end

# replaces generate()+beam_search() numerics (lrcn.jl:585-632,644-678) for a vector of image ids;
# the caller keeps the printing loop of lrcn.jl:633-640 on word_indices = tokens[1:len, i]
function beam_search(net, split, ids, beam_width, nword)
    n = length(ids)
    tokens = zeros(Int64, nword+2, n); lens = zeros(Int32, n); prob = zeros(Float32, n); lps = zeros(Float32, nword+1, n)
    check(ccall((:lrcn_beam_search, lib), Cint,
                (Ptr{Void}, Cint, Ptr{Int64}, Int64, Cint, Cint, Ptr{Int64}, Ptr{Int32}, Ptr{Float32}, Ptr{Float32}),
                net.handle, split, convert(Vector{Int64}, ids), n, beam_width, nword, tokens, lens, prob, lps))
    return [tokens[1:lens[i], i] for i = 1:n], prob, lps
end

# ---- fc7 producer (SURVEY 8 row f-4): replaces get_params_cnn / get_convnet / extract_features (lrcn.jl:190-221, 697-773).
# cnn = the 15 (filter, bias) pairs conv1_1..conv5_3, fc6, fc7 as MatConvNet stores them (filter kh x kw x Cin x Cout,
# bias of Cout values); images = 224 x 224 x 3 x n Float32 from read_image_data (resized, mean subtracted).
function set_cnn!(net, cnn)
    for l = 1:15, which = 0:1
        a = convert(Array{Float32}, cnn[l][which + 1])
        dims = which == 0 ? Int64[size(a,1), size(a,2), size(a,3), size(a,4)] : Int64[length(a), 1, 1, 1]
        check(ccall((:lrcn_set_cnn_param, lib), Cint, (Ptr{Void}, Cint, Cint, Ptr{Float32}, Ptr{Int64}), net.handle, l, which, a, dims))
    end
end
function get_cnn_param(net, l, which, dims)
    a = Array(Float32, dims...)
    check(ccall((:lrcn_get_cnn_param, lib), Cint, (Ptr{Void}, Cint, Cint, Ptr{Float32}, Ptr{Int64}), net.handle, l, which, a,
                convert(Vector{Int64}, collect(dims))))
    return a
end
# relu7 of every image, 4096 x n; normalize=true divides each column by its sum like the featsn files (lrcn.jl:597)
function extract_features(net, images; normalize=true)
    n = size(images, 4); feats = Array(Float32, 4096, n)
    check(ccall((:lrcn_extract_features, lib), Cint, (Ptr{Void}, Ptr{Float32}, Int64, Cint, Ptr{Float32}),
                net.handle, convert(Array{Float32}, images), n, normalize ? 1 : 0, feats))
    return feats
end

# ---- checkpoint sidecar (replaces save(file,"model",model,"vocab",vocab) lrcn.jl:185,230 and load(file) lrcn.jl:88-93).
# Format: include/lrcn_b200.h.  vocab travels as "word\tindex\n" lines.
vocab_bytes(vocab) = convert(Vector{UInt8}, join(["$(w)\t$(i)\n" for (w, i) in sort(collect(vocab), by=last)]))
function vocab_from_bytes(b)
    vocab = Dict{String,Int}()
    for line in split(String(copy(b)), "\n")
        isempty(line) && continue
        k = rsearch(line, '\t'); vocab[line[1:k-1]] = parse(Int, line[k+1:end])
    end
    return vocab
end
function save!(net, path, vocab; with_adam=true)          # weights + Adam m,v,t from the GPU(s) + vocab
    aux = vocab_bytes(vocab)
    check(ccall((:lrcn_checkpoint_save, lib), Cint, (Ptr{Void}, Cstring, Cint, Ptr{UInt8}, Int64), net.handle, path, with_adam ? 1 : 0, aux, length(aux)))
end
function load!(net, path)                                 # -> vocab Dict; restores Adam state when the file has it
    had = Ref{Cint}(0); n = Ref{Int64}(0); aux = zeros(UInt8, filesize(path))
    check(ccall((:lrcn_checkpoint_load, lib), Cint, (Ptr{Void}, Cstring, Ptr{Cint}, Ptr{UInt8}, Int64, Ptr{Int64}), net.handle, path, had, aux, length(aux), n))
    return vocab_from_bytes(aux[1:n[]])
end
# pure-Julia reader of the same file (no library, no GPU): -> (model::Array{Any}(9), vocab, (m, v, t) or nothing),
# e.g. to convert a sidecar back into a .jld with save(file,"model",model,"vocab",vocab)
function read_checkpoint(path)
    open(path) do f
        String(read(f, UInt8, 8)) == "LRCNB2CK" || error("not an LRCNB2CK checkpoint")
        version = read(f, UInt32); flags = read(f, UInt32); dims = read(f, Int32, 4)
        adam_t = read(f, Int64); aux_bytes = read(f, Int64)
        version == 1 || error("unsupported checkpoint version $version")
        function mats()
            out = Array(Any, 9)
            for k = 1:9
                r = read(f, Int64); c = read(f, Int64)
                out[k] = read(f, Float32, (Int(r), Int(c)))          # column-major on disk, like Julia
            end
            return out
        end
        model = mats()
        adam = (flags & 1) == 1 ? (mats(), mats(), adam_t) : nothing
        vocab = vocab_from_bytes(read(f, UInt8, aux_bytes))
        return model, vocab, adam
    end
end

# data-parallel group: rank 0 creates the id, the launcher (MPI.jl / files) distributes it
function comm_unique_id()
    id = zeros(UInt8, 128)
    check(ccall((:lrcn_comm_unique_id, lib), Cint, (Ptr{UInt8},), id)); return id
end
comm_init!(net, id, rank, nranks) = check(ccall((:lrcn_comm_init, lib), Cint, (Ptr{Void}, Ptr{UInt8}, Cint, Cint), net.handle, id, rank, nranks))
# peer-memory exchange: every rank exports a 512-byte blob, the launcher all-gathers them (rank order), every rank imports all
function p2p_export(net)
    blob = zeros(UInt8, 512)
    check(ccall((:lrcn_p2p_export, lib), Cint, (Ptr{Void}, Ptr{UInt8}), net.handle, blob)); return blob
end
p2p_import!(net, blobs::Vector{UInt8}, rank, nranks) = check(ccall((:lrcn_p2p_import, lib), Cint, (Ptr{Void}, Ptr{UInt8}, Cint, Cint), net.handle, blobs, rank, nranks))

sync(net) = check(ccall((:lrcn_sync, lib), Cint, (Ptr{Void},), net.handle))
timer_start(net) = check(ccall((:lrcn_timer_start, lib), Cint, (Ptr{Void},), net.handle))
function timer_stop(net)
    ms = Ref{Float32}(0)
    check(ccall((:lrcn_timer_stop, lib), Cint, (Ptr{Void}, Ptr{Float32}), net.handle, ms)); return ms[]
end

end # module
