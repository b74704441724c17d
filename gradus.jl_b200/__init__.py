"""gradus_b200 -- B200-native geodesic hot path behind Gradus.jl's tracing API.

Host-side mirror (Python, because no Julia toolchain exists in this image) of the slice
of the reference's public API that sits on the per-ray integration path:

    tracegeodesics   (src/tracing/tracing.jl:66-80)
    rendergeodesics  (src/rendering/rendering.jl:28-54)
    lineprofile      (src/line-profiles.jl:121-198, BinningMethod and TransferFunctionMethod)

with the same argument meaning, defaults and error behaviour, and a new ensemble type
`EnsembleB200` next to `EnsembleEndpointThreads` (src/Gradus.jl:412).  All compute goes
through the C ABI of include/gradus_b200.h (libgradus_b200.so, hand-written sm_100a CUDA);
there is no CPU fallback."""
from .api import (  # noqa: F401
    BinningMethod,
    CartesianPlane,
    ConstPointFunctions,
    DatumPlane,
    EnsembleB200,
    EnsembleEndpointThreads,
    GeodesicPoints,
    ImpactParameters,
    GeometricGrid,
    InverseGrid,
    BumblebeeMetric,
    MorrisThorneWormhole,
    DilatonAxion,
    JohannsenMetric,
    JohannsenPsaltisMetric,
    KerrNewmanMetric,
    KerrMetric,
    LinearGrid,
    PolarChart,
    PolarPlane,
    PowerLawEmissivity,
    ShakuraSunyaev,
    StatusCodes,
    TabulatedEmissivity,
    TransferFunctionMethod,
    ThickDisc,
    PolishDoughnut,
    ThinDisc,
    TracingConfiguration,
    EndpointCache,
    HostPointFunction,
    ImageOrder,
    apply,
    apply_point_functions,
    apply_point_functions_batch,
    prerendergeodesics,
    chart_for_metric,
    domain_upper_hemisphere,
    impact_axes,
    inner_radius,
    interpolate_plunging_velocities,
    isco,
    lineprofile,
    rendergeodesics,
    tracegeodesics,
    tracegeodesics_batch,
    tracing_configuration,
    trace_target,
    optimize_for_target,
    impact_parameters_for_target,
)
from . import corona, hostmath, reverberation, tf_integration  # noqa: F401
from ._cabi import GradusB200Error  # noqa: F401
from . import transfer_functions  # noqa: F401
from .transfer_functions import (  # noqa: F401
    CellProber,
    CunninghamTransferData,
    DeviceProber,
    TransferFunctionSetup,
    cunningham_transfer_function,
    cunningham_transfer_functions,
    find_offset_for_radius,
    jacobian_ab_gr,
    transfer_function_table,
)

__version__ = "0.1.0"
