"""Built-in Byzantine clients.  Lookup rule of the reference
(/root/reference/src/blades/simulator.py:127-129): attack name ``x`` ->
module ``attackers.xclient`` -> class ``XClient``."""
from .alieclient import AlieClient
from .ipmclient import IpmClient
from .labelflippingclient import LabelflippingClient
from .minmaxclient import MinmaxClient
from .minsumclient import MinsumClient
from .noiseclient import NoiseClient
from .signflippingclient import SignflippingClient

__all__ = ["AlieClient", "IpmClient", "LabelflippingClient", "MinmaxClient", "MinsumClient", "NoiseClient",
           "SignflippingClient"]
