from .policies import Policy, Policies, PolicyCollection
from .interaction_policies import InteractionPolicies, SocialDistancing
from .close_venue_policies import CloseVenue, CloseVenuePolicies
from .quarantine_policies import Quarantine, QuarantinePolicies
from .regional_policies import (RegionalPolicies, RegionalSocialDistancing, RegionalVenueDistancing,
                                VenuePolicies)
