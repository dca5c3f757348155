# GPPDB200.jl -- the reference-side binding of libgppd.so.
#
# `demodulateall` (reference src/Modulation.jl:344-435) and `buildstates`
# (src/Faint.jl:21-73) as `ccall`s into the B200 library, with the reference's
# signatures, keyword arguments and return types.  How to wire it in (INTEGRATION.md):
#
#   1. copy this file next to src/Modulation.jl and `include("GPPDB200.jl")` from
#      src/GPPupilDemodulation.jl AFTER `include("Modulation.jl")` / `include("Faint.jl")`
#      (the submodule imports the parent's types);
#   2. the submodule's functions are `GPPDB200.demodulateall` / `GPPDB200.buildstates`:
#      they do NOT replace `GPPupilDemodulation.demodulateall` by themselves (a name that
#      is already bound to a function in the parent module cannot be re-declared `const`).
#      Either change the three call sites -- `demodulateall` at
#      src/GPPupilDemodulation.jl:161 and :205, `buildstates` at :144 -- to the qualified
#      names, or delete the Julia bodies (src/Modulation.jl:344-435, src/Faint.jl:21-73)
#      and add `using .GPPDB200: demodulateall, buildstates` after the include.
#
# Error convention = the reference's own FFI idiom (src/FitsUtils.jl:42-58): Cint
# status, error raised on the Julia side.
#
# UNTESTED: no Julia toolchain exists in the build image or on the GPU boxes, so this
# file has never been executed.  The same C ABI (same symbols, argument order and
# buffer layouts) is exercised by the ctypes host mirror
# (gppupildemodulation.jl_b200/api.py) in tests/.
module GPPDB200

import ..GPPupilDemodulation: MetState, FaintStates, Modulation, ModulationWithOffsets,
    ModulationNoOffsets, M_2PI, HIGH, LOW, NORMAL, TRANSIENT

const libgppd = get(ENV, "GPPD_LIBRARY", joinpath(@__DIR__, "libgppd.so"))

const GPPD_ONLYHIGH    = UInt32(1)
const GPPD_FITOFFSETS  = UInt32(2)
const GPPD_NO_RECENTER = UInt32(4)
const GPPD_KEEPRAW     = UInt32(8)
const GPPD_CENTER_EMPIRICAL = UInt32(32)
const GPPD_FP32        = UInt32(64)   # optional reduced-precision harmonic sums (off by default)
const GPPD_CENTER_ELLIPSE = UInt32(128)   # `--center ellipse`: offset + ellipse correction per channel
const GPPD_ELLIPSE_STRIDE = 6

# struct gppd_options (include/gppd.h)
struct Options
    flags::UInt32
    method::Int32
    maxfun::Int32
    has_xinit::Int32
    xinit::NTuple{2,Float64}
    rhobeg::Float64
    rhoend::Float64
    group_mask::UInt32      # 0 = all 8 (telescope, side) groups
    reserved::UInt32
end
Options(flags, method, maxfun, has_xinit, xinit, rhobeg, rhoend) =
    Options(flags, method, maxfun, has_xinit, xinit, rhobeg, rhoend, UInt32(0), UInt32(0))

const handle = Ref{Ptr{Cvoid}}(C_NULL)

function gppd_assert_ok(status::Cint)
    status == 0 && return nothing
    msg = unsafe_string(ccall((:gppd_strerror, libgppd), Cstring, (Cint,), status))
    detail = unsafe_string(ccall((:gppd_last_error, libgppd), Cstring, ()))
    error("libgppd: $msg ($detail)")
end

function gethandle()
    if handle[] == C_NULL
        dev = parse(Int, get(ENV, "GPPD_DEVICE", "0"))
        gppd_assert_ok(ccall((:gppd_create, libgppd), Cint, (Cint, Ref{Ptr{Cvoid}}), dev, handle))
        atexit(() -> ccall((:gppd_destroy, libgppd), Cint, (Ptr{Cvoid},), handle[]))
    end
    return handle[]
end

# buildstates(faintstates, timestamp; lag, preswitchdelay, postwitchdelay), src/Faint.jl:21
function buildstates(faintstates::FaintStates{T,A}, timestamp::AbstractVector;
                     lag::Integer=0, preswitchdelay=0, postwitchdelay=0) where {T<:AbstractFloat,A<:AbstractVector{T}}
    t = convert(Vector{Float64}, timestamp)           # no copy for a Vector{Float64}
    t1 = convert(Vector{Float64}, faintstates.timer1)
    t2 = convert(Vector{Float64}, faintstates.timer2)
    st = Vector{Int8}(undef, length(t))
    gppd_assert_ok(ccall((:gppd_buildstates, libgppd), Cint,
        (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Int64,
         Float64, Float64, Ptr{Int8}),
        gethandle(), length(t), t, t1, length(t1), t2, length(t2), lag,
        Float64(preswitchdelay), Float64(postwitchdelay), st))
    return MetState.(st)
end

# demodulateall(timestamp, data; ...) -> (output, param, likelihood), src/Modulation.jl:344-435
function demodulateall(timestamp::AbstractVector, data::AbstractMatrix{Complex{T}};
                       init::Union{Symbol,Vector{T}}=:auto,
                       recenter::Bool=true,
                       faintparam::Union{Nothing,FaintStates,S}=nothing,
                       onlyhigh=false,
                       fitoffsets=false,
                       preswitchdelay=0.01,
                       postwitchdelay=0.3) where {T<:AbstractFloat,S<:AbstractVector{MetState}}
    n = length(timestamp)
    size(data) == (n, 40) || error("voltage and time must have the same number of lines")
    t = convert(Vector{Float64}, timestamp)           # no copy when the types already match
    d = convert(Matrix{ComplexF64}, data)              # N x 40, column-major (views are copied)
    state = C_NULL
    stvec = Int8[]
    if isa(faintparam, FaintStates)                    # :366-367
        stvec = Int8.(Integer.(buildstates(faintparam, t; preswitchdelay=preswitchdelay,
                                           postwitchdelay=postwitchdelay)))
        state = pointer(stvec)
    elseif !isnothing(faintparam)                      # :368-369
        stvec = Int8.(Integer.(faintparam))
        state = pointer(stvec)
    end
    flags = (onlyhigh ? GPPD_ONLYHIGH : UInt32(0)) | (fitoffsets ? GPPD_FITOFFSETS : UInt32(0)) |
            (recenter ? UInt32(0) : GPPD_NO_RECENTER)
    opt = isa(init, Symbol) ? Options(flags, 0, 0, 0, (0.0, 0.0), 0.0, 0.0) :
                              Options(flags, 0, 0, 1, (Float64(init[1]), Float64(init[2])), 0.0, 0.0)
    output = Matrix{ComplexF64}(undef, n, 40)
    params = Matrix{Float64}(undef, 6, 32)
    chi2 = Vector{Float64}(undef, 32)
    GC.@preserve stvec begin
        gppd_assert_ok(ccall((:gppd_demodulate_f64, libgppd), Cint,
            (Ptr{Cvoid}, Int64, Int64, Ptr{Float64}, Ptr{ComplexF64}, Ptr{Int8}, Ref{Options},
             Ptr{ComplexF64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Float64}),
            gethandle(), n, 0, t, d, state, opt, output, params, chi2, C_NULL, C_NULL))
    end
    if fitoffsets
        param = [ModulationWithOffsets{T}(complex(params[1, i], params[2, i]),
                                          complex(params[3, i], params[4, i]),
                                          params[5, i], params[6, i], M_2PI) for i in 1:32]
    else
        param = [ModulationNoOffsets{T}(complex(params[3, i], params[4, i]),
                                        params[5, i], params[6, i], M_2PI) for i in 1:32]
    end
    return (Matrix{Complex{T}}(output), param, T.(chi2))
end

"""
    processrows!(rows_out, rows, row_bytes, time_off, volt_off, mjd; offsets, faintparam,
                 window, keepraw, onlyhigh) -> (params, chi2, state)

Table-level fast path on the raw bytes of the METROLOGY BINTABLE (big-endian records of
`row_bytes` bytes, TIME at byte `time_off`, VOLT at byte `volt_off`), replacing the array
work of `processmetrology` (src/GPPupilDemodulation.jl:139-171,192-253) and the column
decoding of `Dict(hdu)` (src/FitsUtils.jl:31-37).  `rows_out` receives the output records
(`row_bytes + 256` bytes each with `keepraw`).  `offsets === nothing` fits the centres;
`offsets === true` (processmetrology's default, `--center empirical`) has the library fit
one circle per channel (compute_offsets, :105-125) -- `centres(slot)` returns them;
`offsets === :ellipse` (`--center ellipse`) one ellipse per channel, applied to every row
before the fit -- `ellipses(slot)` returns the maps.
"""
function processrows!(rows_out::Vector{UInt8}, rows::Vector{UInt8}, row_bytes::Integer,
                      time_off::Integer, volt_off::Integer, mjd::Real;
                      offsets::Union{Nothing,Bool,Symbol,Vector{ComplexF64}} = nothing,
                      faintparam::Union{Nothing,FaintStates} = nothing,
                      window::Real = 0.0, keepraw::Bool = false, onlyhigh::Bool = false, slot::Integer = 0,
                      fp32::Bool = false)
    n = length(rows) ÷ row_bytes
    flags = (onlyhigh ? GPPD_ONLYHIGH : UInt32(0)) | (keepraw ? GPPD_KEEPRAW : UInt32(0)) |
            (offsets === true ? GPPD_CENTER_EMPIRICAL : UInt32(0)) | (fp32 ? GPPD_FP32 : UInt32(0)) |
            (offsets === :ellipse ? GPPD_CENTER_ELLIPSE : UInt32(0))
    offsets isa Symbol && offsets !== :ellipse && throw(ArgumentError("offsets: a vector, nothing, true or :ellipse"))
    offsets isa Union{Bool,Symbol} && (offsets = nothing)
    opt = Options(flags, 0, 0, 0, (0.0, 0.0), 0.0, 0.0)
    nwrows = Ref{Int64}(0); nwin = Ref{Int64}(1)
    if window > 0
        t01 = Int32[ntoh(reinterpret(Int32, rows[k*row_bytes+time_off+1:k*row_bytes+time_off+4])[1]) for k in 0:1]
        gppd_assert_ok(ccall((:gppd_table_windows, libgppd), Cint,
            (Int64, Ptr{Int32}, Float64, Float64, Ref{Int64}, Ref{Int64}), 2, t01, mjd, window, nwrows, nwin))
        nwin[] = cld(n, nwrows[])
    end
    params = Matrix{Float64}(undef, 6, 32 * nwin[])
    chi2 = Vector{Float64}(undef, 32 * nwin[])
    state = Vector{Int8}(undef, n)
    t1 = isnothing(faintparam) ? Float64[] : Vector{Float64}(faintparam.timer1)
    t2 = isnothing(faintparam) ? Float64[] : Vector{Float64}(faintparam.timer2)
    GC.@preserve rows rows_out offsets t1 t2 begin
        gppd_assert_ok(ccall((:gppd_submit_fits_rows, libgppd), Cint,
            (Ptr{Cvoid}, Cint, Int64, Ptr{UInt8}, Int64, Int64, Int64, Float64, Ptr{ComplexF64},
             Ptr{Float64}, Int64, Ptr{Float64}, Int64, Float64, Ref{Options}, Ptr{UInt8},
             Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int8}),
            gethandle(), slot, n, rows, row_bytes, time_off, volt_off, mjd,
            isnothing(offsets) ? C_NULL : pointer(offsets), t1, length(t1), t2, length(t2),
            window, opt, rows_out, params, chi2, C_NULL, state))
        gppd_assert_ok(ccall((:gppd_wait, libgppd), Cint, (Ptr{Cvoid}, Cint), gethandle(), slot))
    end
    return (params, chi2, isnothing(faintparam) ? nothing : state)
end

# ---- native file path (include/gppd.h: gppd_file_*) -------------------------------------
# The night loop of src/GPPupilDemodulation.jl:358-392 with the library reading and writing the
# METROLOGY records itself (src/FitsUtils.jl:31-37 and :95-156 on its I/O threads, pinned
# staging, asynchronous copies): Julia keeps the header parsing, the gating and the text of
# the new header.  Ring of `numslots()` files in flight:
#
#     for (i, f) in enumerate(files)
#         s = (i - 1) % nslots
#         i > nslots && finishfile!(s, ...)          # results of the file submitted nslots ago
#         submitfile!(s, f.path, f.data_offset, f.n, f.row_bytes, f.time_off, f.volt_off, f.mjd; ...)
#     end
#     ...finish the remaining slots...;  drainfiles()
const GPPD_SEG_COPY    = Int32(0)   # `length` bytes of the input file from `offset`
const GPPD_SEG_BYTES   = Int32(1)   # `length` bytes from memory (copied at call time)
const GPPD_SEG_RECORDS = Int32(2)   # the output records (+ per-row extra columns), padded to 2880

# struct gppd_file_segment
struct FileSegment
    kind::Int32
    reserved::Int32
    offset::Int64
    length::Int64
    bytes::Ptr{Cvoid}
end
copysegment(offset::Integer, length::Integer) = FileSegment(GPPD_SEG_COPY, 0, offset, length, C_NULL)
recordsegment() = FileSegment(GPPD_SEG_RECORDS, 0, 0, 0, C_NULL)

numslots() = Int(ccall((:gppd_num_slots, libgppd), Cint, (Ptr{Cvoid},), gethandle()))

"""
    submitfile!(slot, path, data_offset, n, row_bytes, time_off, volt_off, mjd; offsets, faintparam,
                window, keepraw, onlyhigh)

Queue one FITS file: `n` METROLOGY records of `row_bytes` bytes start at byte `data_offset` of
`path` (TIME at `time_off`, VOLT at `volt_off` inside a record).  Returns at once.
"""
function submitfile!(slot::Integer, path::AbstractString, data_offset::Integer, n::Integer,
                     row_bytes::Integer, time_off::Integer, volt_off::Integer, mjd::Real;
                     offsets::Union{Nothing,Bool,Symbol,Vector{ComplexF64}} = nothing,
                     faintparam::Union{Nothing,FaintStates} = nothing, window::Real = 0.0,
                     keepraw::Bool = false, onlyhigh::Bool = false)
    flags = (onlyhigh ? GPPD_ONLYHIGH : UInt32(0)) | (keepraw ? GPPD_KEEPRAW : UInt32(0)) |
            (offsets === true ? GPPD_CENTER_EMPIRICAL : UInt32(0)) |
            (offsets === :ellipse ? GPPD_CENTER_ELLIPSE : UInt32(0))
    offsets isa Symbol && offsets !== :ellipse && throw(ArgumentError("offsets: a vector, nothing, true or :ellipse"))
    offsets isa Union{Bool,Symbol} && (offsets = nothing)
    opt = Options(flags, 0, 0, 0, (0.0, 0.0), 0.0, 0.0)
    t1 = isnothing(faintparam) ? Float64[] : Vector{Float64}(faintparam.timer1)
    t2 = isnothing(faintparam) ? Float64[] : Vector{Float64}(faintparam.timer2)
    GC.@preserve offsets t1 t2 begin       # (the library copies all of them before it returns)
        gppd_assert_ok(ccall((:gppd_file_submit, libgppd), Cint,
            (Ptr{Cvoid}, Cint, Cstring, Int64, Int64, Int64, Int64, Int64, Float64, Ptr{ComplexF64},
             Ptr{Float64}, Int64, Ptr{Float64}, Int64, Float64, Ref{Options}),
            gethandle(), slot, path, data_offset, n, row_bytes, time_off, volt_off, mjd,
            isnothing(offsets) ? C_NULL : pointer(offsets), t1, length(t1), t2, length(t2), window, opt))
    end
    return nothing
end

"""
    waitfile(slot, nwin; faint) -> (params 6 x 32 nwin, chi2, state | nothing)

Block until the fits of the slot's file are done (`state` needs the caller to pass the number
of rows through `nrows` when `faint`).
"""
function waitfile(slot::Integer, nwin::Integer = 1; nrows::Integer = 0)
    params = Matrix{Float64}(undef, 6, 32 * nwin)
    chi2 = Vector{Float64}(undef, 32 * nwin)
    state = nrows > 0 ? Vector{Int8}(undef, nrows) : Int8[]
    gppd_assert_ok(ccall((:gppd_file_wait, libgppd), Cint,
        (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int8}),
        gethandle(), slot, params, chi2, C_NULL, nrows > 0 ? pointer(state) : C_NULL))
    return (params, chi2, nrows > 0 ? state : nothing)
end

"""
    writefile!(slot, out_path, segments; extra = nothing, extra_row_bytes = 0)

Queue the output file of the slot's job: the segments in order (`copysegment`, header bytes
as `Vector{UInt8}`, `recordsegment()`).  `extra` (the per-row columns of window mode, one block
of `extra_row_bytes` bytes per row) must stay alive until the slot's next `submitfile!` or
`drainfiles()` returns: the caller keeps the reference.
"""
function writefile!(slot::Integer, out_path::AbstractString, segments::Vector;
                    extra::Union{Nothing,Vector{UInt8}} = nothing, extra_row_bytes::Integer = 0)
    blobs = [s for s in segments if s isa Vector{UInt8}]
    GC.@preserve blobs extra begin
        segs = FileSegment[s isa Vector{UInt8} ?
                           FileSegment(GPPD_SEG_BYTES, 0, 0, length(s), pointer(s)) : s for s in segments]
        gppd_assert_ok(ccall((:gppd_file_write, libgppd), Cint,
            (Ptr{Cvoid}, Cint, Cstring, Ptr{FileSegment}, Int32, Ptr{UInt8}, Int64),
            gethandle(), slot, out_path, segs, length(segs),
            isnothing(extra) ? C_NULL : pointer(extra), extra_row_bytes))
    end
    return nothing
end

"wait for every pending file of the handle; raises the first error"
drainfiles() = gppd_assert_ok(ccall((:gppd_file_drain, libgppd), Cint, (Ptr{Cvoid},), gethandle()))

"centres fitted by the last `offsets = true` call on `slot` (40 complex values)"
function centres(slot::Integer = 0)
    c = Vector{ComplexF64}(undef, 40)
    gppd_assert_ok(ccall((:gppd_centres, libgppd), Cint, (Ptr{Cvoid}, Cint, Int64, Ptr{ComplexF64}),
                         gethandle(), slot, 1, c))
    return c
end

"""
    ellipses(slot = 0) -> (ell, status)

The maps fitted and applied by the last `offsets = :ellipse` call on `slot`: `ell` is a
6 x 40 matrix, column c = (x0, y0, r, alpha, m21, m22) of channel c; `status[c]` is 2
(ellipse), 1 (circle centre, identity shape) or 0 (neither).
"""
function ellipses(slot::Integer = 0)
    ell = Matrix{Float64}(undef, GPPD_ELLIPSE_STRIDE, 40)
    status = Vector{Int32}(undef, 40)
    gppd_assert_ok(ccall((:gppd_ellipses, libgppd), Cint, (Ptr{Cvoid}, Cint, Int64, Ptr{Float64}, Ptr{Int32}),
                         gethandle(), slot, 1, ell, status))
    return ell, status
end

end # module
