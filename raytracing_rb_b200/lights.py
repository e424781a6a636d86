"""Mirror of Alex::Lights::Light / SpotLight (reference src/lights/light.rb:2-11,
src/lights/spot_light.rb:4-5): plain property bags.  SpotLight#intersect? is dead code upstream
(references an undefined `center`) and is not mirrored."""
from ._edits import Tracked


class Light(Tracked):
    position = name = color = high_light_rate = high_light_angle = None

    def __init__(self, properties):  # light.rb:6-10
        for key, value in properties.items():
            setattr(self, key, value)


class SpotLight(Light):
    radius = None


LIGHT_CLASSES = {"Spot": SpotLight}  # world.rb:24 `eval("Alex::Lights::#{type}Light")`
